// k12_union.cu — K12: the k-way term merge finished per bucket (K1b) and the per-term union +
// dedup of uint32 posting lists with the removed filter and the intcomp encoder (K2b).
//
// Replaces
//   - go-iterators' MergingIterator (built at shard.go:267; ordering file.CompareTermValues,
//     file/types.go:24-26): K1b — inside a bucket, equal terms are grouped with a shared-memory
//     hash table and only the DISTINCT terms are ordered (16-byte key windows past the
//     bucket's common prefix; ranked by counting, or a bitonic network when there are many);
//   - file.MergeTermValues (file/types.go:14-22: append + slices.Sort + slices.Compact, applied
//     pairwise), the removed filter of the merge loop (shard.go:181-190) and
//     intcomp.CompressUint32 (file/writer.go:49): K2b — one warp per term, no block barrier:
//     sources gathered into a 1 KB shared-memory slot, sorting network in registers (<= 256
//     values, one shuffle + one predicated min/max per compare-exchange), dedup against the
//     neighbour lane, removed filter (L2-resident bitmap), ballot compaction, encoder run from
//     registers in place, coalesced copy to the term's slot of the `_val` staging buffer.
// Semantics kept bit-exact:
//   - a term present in ONE segment passes through untouched — not sorted, not deduped (survey
//     Q4); a term present in >= 2 segments becomes the sorted-unique union;
//   - the filter runs AFTER the union; removed = membership in the sorted removed list.
// Terms whose lists exceed 256 values are passed on through device-side work lists: up to 1024
// values one warp each (k2_mwarp_kernel), up to 2048 / 4096 one CTA each (k2_medium_kernel<4> /
// <8>, both built on cta_union_term), beyond that the multi-CTA global-memory path at the end of
// this file.  k4_point_kernel (a read of ONE term as one kernel) uses the same CTA union.
// Integer/byte work, HBM-bound by design.
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "intcomp.cuh"
#include "keys.cuh"
#include "union.cuh"
#include "union_dev.cuh"

namespace ii2 {

constexpr int K1B_THREADS = 256;  // a tile holds CAP_I instances: CAP_I / K1B_THREADS per thread
constexpr int K1B_WARPS = K1B_THREADS / 32;
// instances per sub-tile (512 would need k <= 512: a tile holds at least one instance of every segment)
constexpr uint32_t CAP_I = 1024;
constexpr uint32_t K1B_HT = CAP_I > 512 ? 2048 : 1024;  // hash slots (a power of two >= 2 * CAP_I)
static_assert(CAP_I % K1B_THREADS == 0 && CAP_I <= 1024 && CAP_I % 4 == 0,
              "tile = a whole number of instances per thread, 10-bit tile indexes");
constexpr uint32_t K1B_STAGE_CAP = CAP_I * 6;  // postings of a tile assembled in the 24 KB of key windows
constexpr uint32_t K1B_SMALL_D = 64;  // distinct terms ranked by counting instead of sorting
constexpr uint32_t K1B_EMPTY = 0xFFFFFFFFu;
constexpr uint32_t K12_PENDING = 0xFFFFFFFFu;
constexpr uint32_t K1B_HEAVY = 0xFFFFFFFFu;   // pbase of a heavy term

struct K1bArgs {
  const SegDesc* segs;
  int k;
  const uint32_t* part;
  const uint32_t* btb;   // boundary tables of the plan: first term byte / first posting of every run
  const uint64_t* bpo;
  const uint64_t* bk_pos;
  const uint32_t* bk_cpl;
  const uint64_t* bk_P;
  GroupIn* gin;
  uint32_t* gath;   // [N_in] light terms: the sources of a term copied back to back (its slot)
  uint64_t* src_ptr;  // heavy terms only: (pointer, length) of every source
  uint32_t* src_len;
  uint32_t* bk_D;   // [B] distinct terms per bucket
  uint32_t bucket0; // first bucket of this launch (the grid covers a chunk of buckets)
  const uint32_t* list;  // or: the buckets of this launch (those the fused kernel deferred)
};


// Order of two terms whose bytes before `skip` are equal and which both run past `skip`:
// further 16-byte windows until one differs or a term ends.  Kept out of line: the compiler
// must not hoist its offset loads into the callers' fast path.
__device__ __noinline__ int k1b_tail_compare(const SegDesc* __restrict__ segs, int k, uint32_t ix,
                                             uint32_t nx, uint32_t iy, uint32_t ny, uint32_t skip) {
  int sx, sy;
  uint32_t tx, ty;
  locate_instance(segs, k, ix, sx, tx);
  locate_instance(segs, k, iy, sy, ty);
  const SegDesc& dx = segs[sx];
  const SegDesc& dy = segs[sy];
  const uint32_t ox = __ldg(dx.toff + tx);
  const uint32_t oy = __ldg(dy.toff + ty);
  for (uint32_t c = skip;; c += 16) {
    uint64_t hx, lx, hy, ly;
    load_key16(dx.tb, ox, nx, c, hx, lx);
    load_key16(dy.tb, oy, ny, c, hy, ly);
    if (hx != hy) return hx < hy ? -1 : 1;
    if (lx != ly) return lx < ly ? -1 : 1;
    if (!(nx > c + 16 && ny > c + 16)) break;
  }
  return nx < ny ? -1 : (nx > ny ? 1 : 0);
}

__host__ __device__ inline size_t k1b_smem_bytes(int k) {
  return (size_t)CAP_I * 24                      // key_hi, key_lo, key_x
         + (size_t)CAP_I * 4 * 3                 // inst, count|length, pbase
         + (size_t)(4 * k) * 4 + (size_t)(2 * k + 2) * 4   // cur, mm, hi, endr; rstart (padded to 2^n + 1)
         + (size_t)CAP_I * 2 * 2                 // tlen, reps
         + (size_t)k * 40 + 16                   // tb, toff, poff, post pointers; base - lo
         + (size_t)K1B_HT * 4 + 64;
}

constexpr int K1B_MIN_CTAS = 4;
// LIST: the CTA's bucket comes from a.list (the buckets the fused kernel deferred) — a separate
// instantiation, because one more live pointer in the default one costs spills (64 registers).
template <bool LIST>
__global__ void __launch_bounds__(K1B_THREADS, K1B_MIN_CTAS) k1b_group_kernel(const K1bArgs a) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem_raw[];
  __shared__ uint64_t s_ws64[K1B_WARPS + 2];
  __shared__ uint32_t s_ws32[K1B_WARPS + 2];
  __shared__ uint32_t s_nreps, s_tot[2];

  const int k = a.k;
  uint8_t* sp = smem_raw;
  uint64_t* key_hi = reinterpret_cast<uint64_t*>(sp); sp += CAP_I * 8;
  uint64_t* key_lo = reinterpret_cast<uint64_t*>(sp); sp += CAP_I * 8;
  uint64_t* key_x = reinterpret_cast<uint64_t*>(sp); sp += CAP_I * 8;  // bytes 16..23 of the window
  // by representative: sources << 20 | Σ source lengths (each saturated at REG_CAP + 1, so the
  // sum stays below 2^19 for the <= 1024 instances of a tile)
  uint32_t* cg = reinterpret_cast<uint32_t*>(sp); sp += CAP_I * 4;
  uint32_t* inst_a = reinterpret_cast<uint32_t*>(sp); sp += CAP_I * 4;  // global instance id
  // by representative: slot of the term in the bucket's gather region, or K1B_HEAVY
  uint32_t* pbase = reinterpret_cast<uint32_t*>(sp); sp += CAP_I * 4;
  uint16_t* tlen = reinterpret_cast<uint16_t*>(sp); sp += CAP_I * 2;
  uint16_t* reps = reinterpret_cast<uint16_t*>(sp); sp += CAP_I * 2;
  sp += (16 - (reinterpret_cast<uintptr_t>(sp) & 15)) & 15;
  uint32_t* table = reinterpret_cast<uint32_t*>(sp); sp += K1B_HT * 4;  // 16-byte aligned
  uint32_t* cur = reinterpret_cast<uint32_t*>(sp); sp += k * 4;
  uint32_t* mm = reinterpret_cast<uint32_t*>(sp); sp += k * 4;
  uint32_t* hib = reinterpret_cast<uint32_t*>(sp); sp += k * 4;
  uint32_t* endr = reinterpret_cast<uint32_t*>(sp); sp += k * 4;
  // run starts inside the tile, padded with `size` up to kp2 = the power of two >= k
  uint32_t* rstart = reinterpret_cast<uint32_t*>(sp);
  // the segment descriptors of the call, one field per array: phase (2) indexes them by run
  sp += (2 * k + 2) * 4;
  sp += (8 - (reinterpret_cast<uintptr_t>(sp) & 7)) & 7;
  const uint8_t** sg_tb = reinterpret_cast<const uint8_t**>(sp); sp += k * 8;
  const uint32_t** sg_toff = reinterpret_cast<const uint32_t**>(sp); sp += k * 8;
  const uint64_t** sg_poff = reinterpret_cast<const uint64_t**>(sp); sp += k * 8;
  const uint32_t** sg_post = reinterpret_cast<const uint32_t**>(sp); sp += k * 8;
  uint32_t* sg_bl = reinterpret_cast<uint32_t*>(sp);  // base - lo
  // alias, valid once the hash table is done: first source slot by representative
  uint32_t* sbase = table;
  uint32_t kp2 = 1;
  while (kp2 < (uint32_t)k) kp2 <<= 1;

  const uint32_t tid = threadIdx.x;
  const unsigned lane = lane_id(), warp = warp_id();
  const uint32_t b = LIST ? a.list[blockIdx.x] : a.bucket0 + blockIdx.x;
  uint32_t W = (uint32_t)(a.bk_pos[b + 1] - a.bk_pos[b]);
  if (W == 0) {
    if (tid == 0) a.bk_D[b] = 0;
    return;
  }
  {
    const uint32_t r0 = b, r1 = b + 1;
    for (int s = tid; s < k; s += K1B_THREADS) {
      cur[s] = a.part[(uint64_t)r0 * k + s];
      endr[s] = a.part[(uint64_t)r1 * k + s];
      const SegDesc sd = a.segs[s];
      sg_tb[s] = sd.tb;
      sg_toff[s] = sd.toff;
      sg_poff[s] = sd.poff;
      sg_post[s] = sd.post;
      sg_bl[s] = sd.base - sd.lo;
      // the offsets of the run are read in phase (2), a few thousand clocks from here
      asm volatile("prefetch.global.L2 [%0];" ::"l"(sd.toff + cur[s]));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(sd.poff + cur[s]));
      if (endr[s] - cur[s] > 12) asm volatile("prefetch.global.L2 [%0];" ::"l"(sd.poff + endr[s]));
      // (prefetching the run's term bytes and postings here, from the plan's boundary tables,
      // was measured slower than the per-instance prefetches of phase (2): 1.30 vs 1.23 ms, and
      // 1.45 ms with both - the extra live values cost spills at 64 registers)
    }
  }
  const uint64_t rec_base = a.bk_pos[b];
  const uint32_t cpl = a.bk_cpl[b];
  uint32_t* const gath = a.gath + a.bk_P[b];
  uint32_t dcount = 0;   // distinct terms so far in this bucket
  uint32_t icount = 0;   // instances so far
  uint32_t pcount = 0;   // postings of light terms so far
  uint32_t ecount = 0;   // staging words so far
  __syncthreads();

  while (W > 0) {
    // ---------------- choose the sub-tile [cur, mmp) ----------------
    uint32_t size;
    const uint32_t* mmp;   // run ends of the tile
    if (W <= CAP_I) {      // the usual case: the whole (rest of the) bucket is one tile
      mmp = endr;
      size = W;
    } else {
      mmp = mm;
      for (int s = tid; s < k; s += K1B_THREADS) hib[s] = endr[s];
      __syncthreads();
      for (;;) {
        uint64_t best = 0;  // widest run and its median term = pivot
        for (int s = tid; s < k; s += K1B_THREADS) {
          const uint64_t cand = ((uint64_t)(hib[s] - cur[s]) << 32) | (uint32_t)s;
          best = cand > best ? cand : best;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
          const uint64_t o = __shfl_xor_sync(0xffffffffu, best, d);
          best = o > best ? o : best;
        }
        __syncthreads();
        if (lane == 0) s_ws64[warp] = best;
        __syncthreads();
        for (int w2 = 0; w2 < K1B_WARPS; w2++) best = s_ws64[w2] > best ? s_ws64[w2] : best;
        const int spv = (int)(uint32_t)best;
        const uint32_t win = (uint32_t)(best >> 32);  // >= 2: sum of windows > CAP_I >= k
        const uint32_t mid = cur[spv] + (win >> 1);
        const KeyedTerm pivot = keyed_term(a.segs[spv], mid);
        uint32_t part_sum = 0;
        for (int s = tid; s < k; s += K1B_THREADS) {
          const uint32_t m = s == spv ? mid : keyed_lower_bound(a.segs[s], cur[s], hib[s], pivot);
          mm[s] = m;
          part_sum += m - cur[s];
        }
        uint32_t tot;
        block_exclusive_scan(part_sum, s_ws32, tot);
        size = tot;  // >= 1: the pivot's own run contributes mid - cur >= 1
        if (size <= CAP_I) break;
        for (int s = tid; s < k; s += K1B_THREADS) hib[s] = mm[s];
        __syncthreads();
      }
      __syncthreads();
    }

    // ---------------- (1) run starts; reset of the tile state ----------------
    if (k <= 128 && warp != 0) {
      // warp 0 scans; the barrier after the resets below publishes the run starts
    } else if (k <= 128) {
      uint32_t v[4], sum = 0;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int s = lane * 4 + j;
        v[j] = s < k ? mmp[s] - cur[s] : 0u;
        sum += v[j];
      }
      uint32_t ex = warp_inclusive_scan(sum) - sum;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int s = lane * 4 + j;
        if (s < k) rstart[s] = ex;
        ex += v[j];
      }
      for (uint32_t s2 = k + lane; s2 <= kp2; s2 += 32) rstart[s2] = size;
    } else {
      uint32_t run = 0;
      for (int base = 0; base < k; base += K1B_THREADS) {
        const int s = base + tid;
        const uint32_t v = s < k ? mmp[s] - cur[s] : 0u;
        uint32_t tot;
        const uint32_t ex = block_exclusive_scan(v, s_ws32, tot);
        if (s < k) rstart[s] = run + ex;
        run += tot;
      }
      for (uint32_t s2 = k + tid; s2 <= kp2; s2 += K1B_THREADS) rstart[s2] = size;
    }
    for (uint32_t i = tid; i < K1B_HT / 4; i += K1B_THREADS)
      reinterpret_cast<uint4*>(table)[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
    for (uint32_t i = 4 * tid; i < CAP_I; i += 4 * K1B_THREADS)
      *reinterpret_cast<uint4*>(cg + i) = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) s_nreps = 0;
    __syncthreads();

    // bytes past the 24-byte window, only needed for terms longer than cpl+24
    auto tail_compare = [&](uint32_t x, uint32_t y) -> int {
      const uint32_t skip = cpl + 24;
      const uint32_t nx = tlen[x], ny = tlen[y];
      if (nx > skip && ny > skip)
        return k1b_tail_compare(a.segs, k, inst_a[x], nx, inst_a[y], ny, skip);
      return nx < ny ? -1 : (nx > ny ? 1 : 0);
    };
    auto less = [&](uint16_t x, uint16_t y) -> bool {
      const uint64_t hx = key_hi[x], hy = key_hi[y];
      if (hx != hy) return hx < hy;
      const uint64_t lx = key_lo[x], ly = key_lo[y];
      if (lx != ly) return lx < ly;
      const uint64_t xx = key_x[x], xy = key_x[y];
      if (xx != xy) return xx < xy;
      return tail_compare(x, y) < 0;
    };

    // ---------------- (2) key windows + posting lengths ----------------
    constexpr int PER = CAP_I / K1B_THREADS;
    uint64_t pp[PER];   // first posting of the thread's instances
    uint32_t pl[PER];   // their lengths
    uint32_t og[PER];   // representative of their term << 20 | where they go inside its gather slot
    {
      int sg[PER];
      uint32_t ix[PER], to[PER], tn[PER];
      uint64_t p1[PER];
#pragma unroll
      for (int j = 0; j < PER; j++) {
        const uint32_t i = tid + j * K1B_THREADS;
        sg[j] = -1;
        if (i < size) {
          uint32_t lo = 0;  // last s with rstart[s] <= i: the run that holds instance i
          for (uint32_t step = kp2 >> 1; step > 0; step >>= 1)
            if (rstart[lo + step] <= i) lo += step;
          sg[j] = (int)lo;
          ix[j] = cur[lo] + (i - rstart[lo]);
        }
      }
#pragma unroll
      for (int j = 0; j < PER; j++) {
        if (sg[j] >= 0) {
          const uint32_t* const toff_s = sg_toff[sg[j]];
          const uint64_t* const poff_s = sg_poff[sg[j]];
          to[j] = __ldg(toff_s + ix[j]);
          tn[j] = __ldg(toff_s + ix[j] + 1);
          pp[j] = __ldg(poff_s + ix[j]);
          p1[j] = __ldg(poff_s + ix[j] + 1);
        }
      }
#pragma unroll
      for (int j = 0; j < PER; j++)
        if (sg[j] >= 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(sg_tb[sg[j]] + to[j] + cpl));
      // (requesting the words of all four key windows before using any was measured slower,
      // 1.61 vs 1.43 ms, like batching the source copies below: the phase is bound by the
      // L1's handling of these 64-way scattered small reads, not by their latency)
#pragma unroll
      for (int j = 0; j < PER; j++) {
        if (sg[j] >= 0) {
          const uint32_t i = tid + j * K1B_THREADS;
          const uint32_t n = tn[j] - to[j];
          uint64_t kh, kl;
          const uint8_t* const tb_s = sg_tb[sg[j]];
          const uint32_t* const post_s = sg_post[sg[j]];
          const uint32_t inst_s = sg_bl[sg[j]] + ix[j];
          load_key16(tb_s, to[j], n, cpl, kh, kl);
          key_hi[i] = kh;
          key_lo[i] = kl;
          key_x[i] = load_key_x(tb_s, to[j], n, cpl);
          tlen[i] = (uint16_t)n;
          inst_a[i] = inst_s;
          pl[j] = (p1[j] - pp[j]) > 0xFFFFFFFEull ? 0xFFFFFFFFu : (uint32_t)(p1[j] - pp[j]);
          pp[j] = reinterpret_cast<uint64_t>(post_s + pp[j]);
          // the copy of phase (5) is ~15 k clocks away: ask the L2 for the line now
          asm volatile("prefetch.global.L2 [%0];" ::"l"(pp[j]));
        }
      }
    }
    // a thread's keys are visible to the block before it enters the hash table: whoever finds
    // its slot taken reads the owner's keys after the CAS
    __threadfence_block();

    // ---------------- (3) group equal terms (hash table of representatives) ----------------
#pragma unroll
    for (int j = 0; j < PER; j++) {
      const uint32_t i = tid + j * K1B_THREADS;
      if (i >= size) break;
      const uint64_t kh = key_hi[i], kl = key_lo[i];
      // four 32-bit multiplies folded together; the top bits pick the slot
      uint32_t h = (uint32_t)kh * 0x9E3779B1u ^ (uint32_t)(kh >> 32) * 0x85EBCA77u ^
                   (uint32_t)kl * 0xC2B2AE3Du ^ (uint32_t)(kl >> 32) * 0x27D4EB2Fu;
      h = (h ^ (h >> 15)) * 0x2C1B3C6Du + tlen[i];
      uint32_t slot = (h ^ (h >> 13)) & (K1B_HT - 1);
      uint32_t rep;
      for (;;) {
        const uint32_t prev = atomicCAS(&table[slot], K1B_EMPTY, i);
        if (prev == K1B_EMPTY) {
          rep = i;
          reps[atomicAdd(&s_nreps, 1u)] = (uint16_t)i;
          break;
        }
        if (*(volatile uint64_t*)&key_hi[prev] == kh && *(volatile uint64_t*)&key_lo[prev] == kl &&
            *(volatile uint16_t*)&tlen[prev] == tlen[i] &&
            *(volatile uint64_t*)&key_x[prev] == key_x[i] && tail_compare(i, prev) == 0) {
          rep = prev;
          break;
        }
        slot = (slot + 1) & (K1B_HT - 1);
      }
      // Σ source lengths, saturating per source so the sum cannot wrap: heavy iff sum > REG_CAP.
      // For a light term every addend is exact, so the value before the add is where this
      // source starts inside the term's gather slot.
      og[j] = (rep << 20) |
              (atomicAdd(&cg[rep], (1u << 20) | (pl[j] > REG_CAP ? REG_CAP + 1 : pl[j])) & 0xFFFFFu);
    }
    __syncthreads();
    const uint32_t D = s_nreps;

    // ---------------- (4) order the distinct terms; one record per term ----------------
    if (D <= K1B_SMALL_D) {  // rank by counting: EIGHT lanes per term, four terms per warp
      // (a warp per term leaves most lanes idle at ~24 distinct terms per bucket and takes
      // three rounds: 1.26 -> 1.23 ms; a thread per term issues a ninth of the instructions
      // and was measured SLOWER, 1.37 vs 1.29 ms: the serial loop sits on the tile's critical
      // path while seven warps wait at the barrier)
      const unsigned sub = lane & 7u;
#pragma unroll 1
      for (uint32_t t0 = warp * 4; t0 < D; t0 += K1B_WARPS * 4) {
        const uint32_t t = t0 + (lane >> 3);
        const bool valid = t < D;
        const uint32_t me = valid ? reps[t] : 0u;
        uint32_t rank = 0, ib = 0, pst = 0, est = 0;
        if (valid) {
          const uint64_t mh = key_hi[me], ml = key_lo[me], mx = key_x[me];
#pragma unroll 1
          for (uint32_t j = sub; j < D; j += 8) {
            const uint32_t o = reps[j];
            const uint64_t oh = key_hi[o];
            bool lt = oh < mh;
            if (oh == mh && o != me) {  // rare: the first eight bytes past the prefix agree
              const uint64_t ol = key_lo[o], ox = key_x[o];
              lt = ol != ml ? ol < ml : (ox != mx ? ox < mx : tail_compare(o, me) < 0);
            }
            const uint32_t c = cg[o];
            const uint32_t len = c & 0xFFFFFu;
            const bool lg = lt && len <= REG_CAP;
            rank += lt ? 1u : 0u;
            ib += lt ? c >> 20 : 0u;
            pst += lg ? len : 0u;
            est += lg ? enc_slot_words(len) : 0u;
          }
        }
#pragma unroll
        for (int d = 4; d > 0; d >>= 1) {
          rank += __shfl_xor_sync(0xffffffffu, rank, d);
          ib += __shfl_xor_sync(0xffffffffu, ib, d);
          pst += __shfl_xor_sync(0xffffffffu, pst, d);
          est += __shfl_xor_sync(0xffffffffu, est, d);
        }
        if (valid && sub == 0) {
          const uint32_t cme = cg[me];
          const uint32_t len = cme & 0xFFFFFu;
          const bool light = len <= REG_CAP;
          const uint32_t src = (uint32_t)rec_base + icount + ib;
          uint4* rec = reinterpret_cast<uint4*>(a.gin + rec_base + dcount + rank);
          rec[0] = make_uint4(inst_a[me], tlen[me], src, cme >> 20);
          rec[1] = make_uint4(len, pcount + pst, ecount + est, 0u);
          sbase[me] = src;
          pbase[me] = light ? pcount + pst : K1B_HEAVY;
          if (rank == D - 1) {
            s_tot[0] = pst + (light ? len : 0u);
            s_tot[1] = est + (light ? enc_slot_words(len) : 0u);
          }
        }
      }
    } else {
      bitonic_sort_any(reps, D, tid, (uint32_t)K1B_THREADS, less, [] { __syncthreads(); });
      __syncthreads();
      uint32_t run_i = 0, run_p = 0, run_e = 0;
      for (uint32_t base = 0; base < D; base += K1B_THREADS) {
        const uint32_t r = base + tid;
        uint32_t me = 0, ci = 0, li = 0, ei = 0;
        uint32_t len = 0;
        if (r < D) {
          me = reps[r];
          ci = cg[me] >> 20;
          len = cg[me] & 0xFFFFFu;
          if (len <= REG_CAP) {
            li = len;
            ei = enc_slot_words(li);
          }
        }
        uint32_t ti, tp, te;
        const uint32_t xi = block_exclusive_scan(ci, s_ws32, ti);
        const uint32_t xp = block_exclusive_scan(li, s_ws32, tp);
        const uint32_t xe = block_exclusive_scan(ei, s_ws32, te);
        if (r < D) {
          GroupIn g;
          g.inst = inst_a[me];
          g.tlen = tlen[me];
          g.src = (uint32_t)rec_base + icount + run_i + xi;
          g.c = ci;
          g.L = len;
          g.pst = pcount + run_p + xp;
          g.eslot = ecount + run_e + xe;
          g.pad = 0;
          a.gin[rec_base + dcount + r] = g;
          sbase[me] = g.src;
          pbase[me] = len <= REG_CAP ? g.pst : K1B_HEAVY;
        }
        run_i += ti;
        run_p += tp;
        run_e += te;
      }
      if (tid == 0) {
        s_tot[0] = run_p;
        s_tot[1] = run_e;
      }
    }
    __syncthreads();

    // ---------------- (5) sources of every term ---------------------------------------------
    // light terms: the postings themselves, copied into the term's slot (any order: the union
    // sorts; a single-source term is one copy, order kept); heavy terms: (pointer, length).
    // A source lands in the middle of its term's slot, so stored straight to global memory the
    // lanes of a warp hit 32 different lines per store (ncu: the LSU data pipe is the busiest
    // unit of this kernel, 60 % of its wavefront peak, a third of it these stores).  The slots of
    // one tile are contiguous in the bucket's gather region: the tile is assembled in shared
    // memory (the key windows are dead by now) and written out as one coalesced stream.
    // (requesting the first values of all four sources before storing any was measured
    // slower: 1.59 vs 1.44 ms)
    const uint32_t tile_p = s_tot[0];
    const bool staged = tile_p <= K1B_STAGE_CAP;
    uint32_t* const stage = reinterpret_cast<uint32_t*>(key_hi);  // key_hi | key_lo | key_x
    auto copy_source = [](const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, uint32_t n) {
      uint32_t t = 0;
#pragma unroll 1
      for (; t + 4 <= n; t += 4) {  // loads first: four in flight per thread
        const uint32_t x0 = __ldg(src + t), x1 = __ldg(src + t + 1), x2 = __ldg(src + t + 2),
                       x3 = __ldg(src + t + 3);
        dst[t] = x0;
        dst[t + 1] = x1;
        dst[t + 2] = x2;
        dst[t + 3] = x3;
      }
      if (t < n) {
        const uint32_t x0 = __ldg(src + t);
        const uint32_t x1 = t + 1 < n ? __ldg(src + t + 1) : 0u;
        const uint32_t x2 = t + 2 < n ? __ldg(src + t + 2) : 0u;
        dst[t] = x0;
        if (t + 1 < n) dst[t + 1] = x1;
        if (t + 2 < n) dst[t + 2] = x2;
      }
    };
#pragma unroll
    for (int j = 0; j < PER; j++) {
      const uint32_t i = tid + j * K1B_THREADS;
      if (i < size) {
        const uint32_t g = og[j] >> 20;
        const uint32_t pb = pbase[g];
        if (pb != K1B_HEAVY) {
          const uint32_t* src = reinterpret_cast<const uint32_t*>(pp[j]);
          const uint32_t at = pb + (og[j] & 0xFFFFFu);
          if (staged)
            copy_source(src, stage + (at - pcount), pl[j]);
          else
            copy_source(src, gath + at, pl[j]);
        } else {
          const uint32_t at = sbase[g] + ((atomicSub(&cg[g], 1u << 20) >> 20) - 1u);
          a.src_ptr[at] = pp[j];
          a.src_len[at] = pl[j];
        }
      }
    }
    if (staged) {
      __syncthreads();
      uint32_t* const out = gath + pcount;
      // head up to the first 16-byte boundary of the destination, then 128-bit stores
      const uint32_t head = min(tile_p, (uint32_t)((16u - ((uintptr_t)out & 15u)) & 15u) >> 2);
      if (tid < head) out[tid] = stage[tid];
      const uint32_t nvec = (tile_p - head) >> 2;
      for (uint32_t v = tid; v < nvec; v += K1B_THREADS) {
        const uint32_t e = head + 4 * v;
        *reinterpret_cast<uint4*>(out + e) =
            make_uint4(stage[e], stage[e + 1], stage[e + 2], stage[e + 3]);
      }
      const uint32_t tail0 = head + 4 * nvec;
      if (tail0 + tid < tile_p) out[tail0 + tid] = stage[tail0 + tid];
    }
    dcount += D;
    icount += size;
    pcount += s_tot[0];
    ecount += s_tot[1];
    W -= size;
    if (W == 0) break;
    __syncthreads();
    for (int s = tid; s < k; s += K1B_THREADS) cur[s] = mmp[s];
    __syncthreads();
  }
  if (tid == 0) a.bk_D[b] = dcount;
}


// ---------------------------------------------------------------- K2b: two terms per warp
constexpr int K2B_THREADS = 128;
constexpr int K2B_WARPS = K2B_THREADS / 32;
constexpr uint32_t K2B_HALF = 128;  // a 16-lane group handles terms of fewer values than this
constexpr uint32_t K2B_ENC_WORDS = 3 + 2 * 129 + 1 + (5 * 127 + 3) / 4 + 1;  // enc_bound(255)
constexpr uint32_t K2B_EBUF = (K2B_ENC_WORDS + 7) & ~7u;  // per warp; a half gets half of it
static_assert(K2B_EBUF / 2 >= 1 + (5 * 127 + 3) / 4, "var-byte stream of 127 values fits a half");

struct K2bArgs {
  const uint64_t* bk_pos;
  const uint64_t* bk_P;
  const uint64_t* bk_E;   // exclusive prefixes of the staging words
  const uint32_t* bk_D;
  const GroupIn* gin;
  RemovedSet rem;
  int want_enc, want_dec, keep_empty;
  GroupRec* recs;
  uint32_t* gath;     // gather slots filled by K1b; the decoded result replaces them in place
  uint32_t* tmp_enc;
  uint64_t* bk_raw;  // [4][nb1], zeroed
  uint32_t nb1;
  uint32_t* n_large;
  uint32_t* large_rec;
  uint32_t* large_bucket;
  uint32_t bucket0;  // first bucket of this launch
  const uint32_t* list;  // or: the buckets of this launch
};

constexpr int K2B_MIN_CTAS = 8;
template <bool LIST>
__global__ void __launch_bounds__(K2B_THREADS, K2B_MIN_CTAS) k2b_union_kernel(const K2bArgs a) {
  pdl_enter();
  __shared__ __align__(16) uint32_t s_buf[K2B_WARPS][REG_CAP];
  __shared__ __align__(16) uint32_t s_enc[K2B_WARPS][K2B_EBUF];
  const unsigned lane = lane_id(), warp = warp_id();
  const unsigned half = lane >> 4, hl = lane & 15u;
  const uint32_t b = LIST ? a.list[blockIdx.x] : a.bucket0 + blockIdx.x;
  const uint32_t D = a.bk_D[b];
  if (D == 0) return;
  const uint64_t rec_base = a.bk_pos[b];
  uint32_t* const gath = a.gath + a.bk_P[b];
  uint32_t* const enc_base = a.tmp_enc + a.bk_E[b];
  uint32_t acc_t = 0, acc_tb = 0, acc_e = 0;  // per group leader (hl == 0) and warp leader
  uint64_t acc_p = 0;
  const GroupIn g_none = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  GroupIn g_next = g_none;
  if (2 * warp + half < D) g_next = a.gin[rec_base + 2 * warp + half];
#pragma unroll 1
  for (uint32_t p0 = 2 * warp; p0 < D; p0 += 2 * K2B_WARPS) {
    // ---- the pair of terms of this warp: one per 16-lane group ----
    const uint32_t r = p0 + half;
    const bool has = r < D;
    const GroupIn g = g_next;
    {  // the record of the next round: in flight while this one is processed
      const uint32_t rn = r + 2 * K2B_WARPS;
      g_next = g_none;
      if (rn < D) g_next = a.gin[rec_base + rn];
    }

    const bool heavy = has && g.L > REG_CAP;
    const bool wide = has && !heavy && g.L >= K2B_HALF;
    if (heavy && hl == 0) {  // the multi-CTA path works from the source list
      const uint32_t slot = atomicAdd(a.n_large, 1u);
      a.large_rec[slot] = (uint32_t)(rec_base + r);
      a.large_bucket[slot] = b;
      GroupRec rec;
      rec.inst = g.inst;
      rec.tlen = g.tlen;
      rec.dec = 0;
      rec.eoff = 0;
      rec.enc = 0;
      rec.cnt = K12_PENDING;
      a.recs[rec_base + r] = rec;
    }
    {
      const bool mine = has && !heavy && !wide;
      const uint32_t L = mine ? g.L : 0u;
      uint32_t* const slot = gath + g.pst;
      uint32_t* const buf = s_buf[warp] + half * K2B_HALF;
      uint32_t* const ebuf = s_enc[warp] + half * (K2B_EBUF / 2);
      const uint32_t outn = union_blocked<16>(slot, buf, L, g.c > 1, a.rem);
      if (a.want_dec)
        for (uint32_t e = hl; e < outn; e += 16) slot[e] = buf[e];
      uint32_t enc = 0;
      uint32_t* const enc_dst = enc_base + g.eslot;
      if (a.want_enc) {
        enc = encode_small_blocked<16>(buf, outn, ebuf);
        for (uint32_t e = hl; e < enc; e += 16) enc_dst[e] = ebuf[e];
      }
      if (mine && hl == 0) {
        GroupRec rec;
        rec.inst = g.inst;
        rec.tlen = g.tlen;
        rec.dec = reinterpret_cast<uint64_t>(slot);
        rec.eoff = a.want_enc ? reinterpret_cast<uint64_t>(enc_dst) : 0ull;
        rec.cnt = outn;
        rec.enc = enc;
        a.recs[rec_base + r] = rec;
        if (outn || a.keep_empty) {
          acc_t += 1;
          acc_tb += g.tlen;
          acc_p += outn;
          acc_e += enc;
        }
      }
      __syncwarp();
    }
    // ---- terms of 128 .. 256 values: the whole warp, one after the other ----
    unsigned wmask = __ballot_sync(0xffffffffu, wide && hl == 0);
    while (wmask) {
      const int src = __ffs(wmask) - 1;  // lane 0 or 16: leader of the group that owns the term
      wmask &= wmask - 1;
      GroupIn w;
      w.inst = __shfl_sync(0xffffffffu, g.inst, src);
      w.tlen = __shfl_sync(0xffffffffu, g.tlen, src);
      w.c = __shfl_sync(0xffffffffu, g.c, src);
      w.L = __shfl_sync(0xffffffffu, g.L, src);
      w.pst = __shfl_sync(0xffffffffu, g.pst, src);
      w.eslot = __shfl_sync(0xffffffffu, g.eslot, src);
      const uint32_t rw = p0 + (src >> 4);
      uint32_t* const slot = gath + w.pst;
      uint32_t* const buf = s_buf[warp];
      uint32_t* const ebuf = s_enc[warp];
      const uint32_t outn = union_blocked<32>(slot, buf, w.L, w.c > 1, a.rem);
      if (a.want_dec)
        for (uint32_t e = lane; e < outn; e += 32) slot[e] = buf[e];
      uint32_t enc = 0;
      uint32_t* const enc_dst = enc_base + w.eslot;
      if (a.want_enc && outn) {
        enc = encode_shared_warp(buf, outn, ebuf);
        for (uint32_t e = lane; e < enc; e += 32) enc_dst[e] = ebuf[e];
      }
      if (lane == 0) {
        GroupRec rec;
        rec.inst = w.inst;
        rec.tlen = w.tlen;
        rec.dec = reinterpret_cast<uint64_t>(slot);
        rec.eoff = a.want_enc ? reinterpret_cast<uint64_t>(enc_dst) : 0ull;
        rec.cnt = outn;
        rec.enc = enc;
        a.recs[rec_base + rw] = rec;
        if (outn || a.keep_empty) {
          acc_t += 1;
          acc_tb += w.tlen;
          acc_p += outn;
          acc_e += enc;
        }
      }
      __syncwarp();
    }
  }
  if (hl == 0 && acc_t) {
    unsigned long long* bo = reinterpret_cast<unsigned long long*>(a.bk_raw);
    atomicAdd(&bo[0ull * a.nb1 + b], (unsigned long long)acc_t);
    atomicAdd(&bo[1ull * a.nb1 + b], (unsigned long long)acc_tb);
    atomicAdd(&bo[2ull * a.nb1 + b], (unsigned long long)acc_p);
    atomicAdd(&bo[3ull * a.nb1 + b], (unsigned long long)acc_e);
  }
}

// ---------------------------------------------------------------- mid terms (one WARP each)
// Terms of REG_CAP < L <= MW_CAP (1024) values: 32 values per lane in registers (union_dev.cuh,
// sort_warp_v<32>: about two warp instructions per value), no block barrier anywhere — the
// K2b design one size up.  The warps pull terms from the list K2b filled (device-side ticket);
// longer terms go on to the CTA-per-term kernel below.
constexpr uint32_t MW_CAP = 1024;
constexpr int MW_V = 32;
constexpr int MW_WARPS = 4;
constexpr int MW_MIN_CTAS = 5;  // 96 registers (6 = 80 registers measured no faster)
constexpr uint32_t MW_BUF = MW_CAP + MW_CAP / 32 + 8;   // one pad word per 32 values (bank-conflict-free blocked loads)
constexpr uint32_t MW_EBUF = 3 + 8 * 129 + 1 + 1 + 6;   // enc_bound(1024) (also holds the source prefix: c + 1 <= 1025 entries)
static_assert(MW_EBUF >= kMaxSegs + 1, "source prefix fits the stream buffer");

struct MwArgs {
  const uint32_t* n_in_list;     // terms K2b deferred
  const uint32_t* in_rec;
  const uint32_t* in_bucket;
  const GroupIn* gin;
  const uint64_t* src_ptr;
  const uint32_t* src_len;
  GroupRec* recs;
  RemovedSet rem;
  int want_enc, keep_empty;
  uint64_t* bk_raw;
  uint32_t nb1;
  uint32_t* cursor;              // next item
  uint32_t* n_out_list;          // terms passed on (> MW_CAP values)
  uint32_t* out_rec;
  uint32_t* out_bucket;
  uint32_t* out_post;
  uint32_t* out_enc;
  unsigned long long* out_cursor;  // [0] postings, [1] words
};

__global__ void __launch_bounds__(MW_WARPS * 32, MW_MIN_CTAS) k2_mwarp_kernel(const MwArgs a) {
  pdl_enter();
  __shared__ __align__(16) uint32_t s_buf[MW_WARPS][MW_BUF];
  __shared__ __align__(16) uint32_t s_enc[MW_WARPS][MW_EBUF];
  const unsigned lane = lane_id(), warp = warp_id();
  uint32_t* const buf = s_buf[warp];
  uint32_t* const ebuf = s_enc[warp];
  uint32_t* const moff = ebuf;  // prefix of the source lengths, dead before the encoder runs
  for (;;) {
    uint32_t item = 0;
    if (lane == 0) item = atomicAdd(a.cursor, 1u);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= *a.n_in_list) return;
    const uint32_t rec = a.in_rec[item], bucket = a.in_bucket[item];
    const GroupIn g = a.gin[rec];
    const uint32_t c = g.c, beg = g.src;
    // ---- source lengths -> prefix (saturating); L
    uint32_t run = 0;
    for (uint32_t base = 0; base < c; base += 32) {
      const uint32_t i = base + lane;
      uint32_t li = i < c ? a.src_len[beg + i] : 0u;
      li = li > MW_CAP + 1 ? MW_CAP + 1 : li;
      const uint32_t inc = warp_inclusive_scan(li);
      if (i < c) moff[i] = min(run + inc - li, MW_CAP + 1);
      run = min(run + __shfl_sync(0xffffffffu, inc, 31), MW_CAP + 1);
    }
    if (run > MW_CAP) {  // uniform: leave it to the CTA-per-term kernel
      if (lane == 0) {
        const uint32_t at = atomicAdd(a.n_out_list, 1u);
        a.out_rec[at] = rec;
        a.out_bucket[at] = bucket;
      }
      continue;
    }
    const uint32_t L = run;
    __syncwarp();
    // ---- gather (element e lives at e + e / 32: padded blocks).  The lanes fetch 32 source
    // descriptors at once; the sources are then copied four at a time (64 values of each), their loads
    // issued before any store, so a term of 32 sources costs ~9 memory round trips instead of 64
    // dependent ones
    for (uint32_t base = 0; base < c; base += 32) {
      const uint32_t j = base + lane;
      uint64_t my_p = 0;
      uint32_t my_o = 0, my_n = 0;
      if (j < c) {
        my_p = a.src_ptr[beg + j];
        my_o = moff[j];
        my_n = (j + 1 < c ? moff[j + 1] : L) - my_o;
      }
      const uint32_t cnt = min(32u, c - base);
      for (uint32_t j0 = 0; j0 < cnt; j0 += 4) {
        uint32_t x[4][2], o4[4], n4[4];
        const uint32_t* p4[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int sl = (int)(j0 + q) & 31;
          p4[q] = reinterpret_cast<const uint32_t*>(__shfl_sync(0xffffffffu, my_p, sl));
          o4[q] = __shfl_sync(0xffffffffu, my_o, sl);
          n4[q] = j0 + q < cnt ? __shfl_sync(0xffffffffu, my_n, sl) : 0u;
          x[q][0] = lane < n4[q] ? __ldg(p4[q] + lane) : 0u;
          x[q][1] = 32 + lane < n4[q] ? __ldg(p4[q] + 32 + lane) : 0u;
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
#pragma unroll
          for (int h = 0; h < 2; h++)
            if (h * 32 + lane < n4[q]) {
              const uint32_t e = o4[q] + h * 32 + lane;
              buf[e + (e >> 5)] = x[q][h];
            }
          // sources of more than 64 values: four loads in flight per lane
          for (uint32_t t0 = 64 + lane; t0 < n4[q]; t0 += 128) {
            uint32_t y[4];
#pragma unroll
            for (int h = 0; h < 4; h++) y[h] = t0 + h * 32 < n4[q] ? __ldg(p4[q] + t0 + h * 32) : 0u;
#pragma unroll
            for (int h = 0; h < 4; h++)
              if (t0 + h * 32 < n4[q]) {
                const uint32_t e = o4[q] + t0 + h * 32;
                buf[e + (e >> 5)] = y[h];
              }
          }
        }
      }
    }
    __syncwarp();
    uint32_t v[MW_V];
#pragma unroll
    for (int r = 0; r < MW_V; r++) {
      const uint32_t e = lane * MW_V + r;
      v[r] = e < L ? buf[lane * (MW_V + 1) + r] : 0xFFFFFFFFu;
    }
    const bool multi = c > 1;  // a single source passes through unsorted, duplicates kept (Q4)
    if (multi) sort_warp_v<MW_V>(v, lane, L);
    // ---- removed filter (eight probes in flight at a time), dedup against the predecessor
    uint32_t keep = 0;
    if (a.rem.bitmap) {
      const uint32_t nbits = (uint32_t)a.rem.bitmap_bits;
#pragma unroll
      for (int r0 = 0; r0 < MW_V; r0 += 8) {
        uint32_t word[8];
#pragma unroll
        for (int r = 0; r < 8; r++) {
          const bool probe = lane * MW_V + r0 + r < L && v[r0 + r] < nbits;
          word[r] = probe ? __ldg(a.rem.bitmap + (v[r0 + r] >> 5)) : 0u;
        }
#pragma unroll
        for (int r = 0; r < 8; r++)
          keep |= (lane * MW_V + r0 + r < L && !((word[r] >> (v[r0 + r] & 31u)) & 1u)) ? 1u << (r0 + r) : 0u;
      }
    } else {
#pragma unroll
      for (int r = 0; r < MW_V; r++)
        if (lane * MW_V + r < L && !(a.rem.n && is_removed_call(a.rem.sorted, a.rem.n, v[r]))) keep |= 1u << r;
    }
    const uint32_t up = __shfl_up_sync(0xffffffffu, v[MW_V - 1], 1);
    if (multi) {
      if (lane > 0 && up == v[0]) keep &= ~1u;
#pragma unroll
      for (int r = 1; r < MW_V; r++)
        if (v[r] == v[r - 1]) keep &= ~(1u << r);
    }
    const uint32_t cnt = __popc(keep);
    const uint32_t inc = warp_inclusive_scan(cnt);
    const uint32_t outn = __shfl_sync(0xffffffffu, inc, 31);
    __syncwarp();  // every lane holds its values: the buffer can be rewritten, dense this time
    {
      uint32_t* dst = buf + (inc - cnt);
#pragma unroll
      for (int r = 0; r < MW_V; r++) {
        const bool k = (keep >> r) & 1u;
        if (k) *dst = v[r];
        dst += k ? 1 : 0;
      }
    }
    __syncwarp();
    // ---- output space, stream, values, record
    unsigned long long pos_p = 0, pos_e = 0;
    if (lane == 0) {
      pos_p = atomicAdd(&a.out_cursor[0], (unsigned long long)outn);
      if (a.want_enc) pos_e = atomicAdd(&a.out_cursor[1], (unsigned long long)intcomp::enc_bound(outn));
    }
    pos_p = __shfl_sync(0xffffffffu, pos_p, 0);
    pos_e = __shfl_sync(0xffffffffu, pos_e, 0);
    uint32_t* const dst_post = a.out_post + pos_p;
    uint32_t* const dst_enc = a.out_enc + pos_e;
    for (uint32_t e = lane; e < outn; e += 32) dst_post[e] = buf[e];
    uint32_t enc = 0;
    if (a.want_enc && outn) {
      enc = encode_shared_warp(buf, outn, ebuf);
      for (uint32_t e = lane; e < enc; e += 32) dst_enc[e] = ebuf[e];
    }
    if (lane == 0) {
      GroupRec& r = a.recs[rec];
      r.cnt = outn;
      r.enc = enc;
      r.dec = reinterpret_cast<uint64_t>(dst_post);
      r.eoff = reinterpret_cast<uint64_t>(dst_enc);
      if (outn || a.keep_empty) {
        unsigned long long* bo = reinterpret_cast<unsigned long long*>(a.bk_raw);
        atomicAdd(&bo[0ull * a.nb1 + bucket], 1ull);
        atomicAdd(&bo[1ull * a.nb1 + bucket], (unsigned long long)r.tlen);
        atomicAdd(&bo[2ull * a.nb1 + bucket], (unsigned long long)outn);
        atomicAdd(&bo[3ull * a.nb1 + bucket], (unsigned long long)enc);
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------- medium terms (one CTA each)
// Terms of REG_CAP < L <= 4096 values — every term of an index with ~1000 postings per term,
// the head of a Zipf distribution — used to take the multi-kernel global-memory path below: a
// host round trip for the lengths, a gather pass, a tile sort pass and a finish pass over the
// same values.  Here one CTA unions a term entirely in shared memory: sources gathered by
// binary search over their length prefix (or a warp per source), runs of 512 values sorted in
// registers (one warp each, sort_warp_v<16>), up to three bitonic merge levels whose cross-warp
// stages go through shared memory, dedup + removed filter + compaction from the registers,
// whole-CTA intcomp encode, one write of the result.  The CTAs pull terms from the
// list K2b filled (a device-side counter: no host synchronisation); output space comes from two
// bump cursors over regions sized by the input postings.  Longer terms go on to the `huge`
// list for the path below.  The union itself is cta_union_term (union_dev.cuh).

struct MedArgs {
  const uint32_t* n_large;       // terms K2b deferred
  const uint32_t* large_rec;
  const uint32_t* large_bucket;
  const GroupIn* gin;
  const uint64_t* src_ptr;
  const uint32_t* src_len;
  GroupRec* recs;
  RemovedSet rem;
  int want_enc, keep_empty;
  uint64_t* bk_raw;
  uint32_t nb1;
  uint32_t* cursor;              // next item of the list
  uint32_t* n_huge;              // terms left to the multi-CTA path
  uint32_t* huge_rec;
  uint32_t* huge_bucket;
  uint32_t* out_post;            // unions, bump-allocated
  uint32_t* out_enc;             // `_val` streams, bump-allocated (upper-bound slots)
  unsigned long long* out_cursor;  // [0] postings, [1] words
};

template <int NW>
__global__ void __launch_bounds__(NW * 32, NW == 4 ? 8 : 5) k2_medium_kernel(const MedArgs a) {
  pdl_enter();
  constexpr int MED_THREADS = NW * 32;
  constexpr uint32_t MED_CAP = NW * MED_RUN;  // values one CTA of NW warps unions
  __shared__ uint32_t s_v[MED_CAP];                 // source pointers / exchange buffer / survivors
  __shared__ uint32_t s_o[MED_CAP + MED_CAP / 16];  // gathered values (padded runs) / exchange buffer
  __shared__ uint32_t s_moff[kMaxSegs + 1];    // prefix of the source lengths
  __shared__ uint64_t s_ws[MED_THREADS / 32 + 2];
  __shared__ uint32_t s_stage[(MED_THREADS / 32) * intcomp::kStageWords];
  __shared__ uint32_t s_table[MED_CAP / 128 + 1];
  __shared__ uint32_t s_item;
  __shared__ uint32_t s_cnt[MED_THREADS / 32];
  __shared__ uint32_t s_last[MED_THREADS / 32];
  __shared__ unsigned long long s_pos[2];
  const uint32_t tid = threadIdx.x;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_item = atomicAdd(a.cursor, 1u);
    __syncthreads();
    const uint32_t item = s_item;
    if (item >= *a.n_large) return;
    const uint32_t rec = a.large_rec[item], bucket = a.large_bucket[item];
    const GroupIn g = a.gin[rec];
    const uint32_t c = g.c, beg = g.src;
    // ---- source lengths -> prefix; total L (saturating: anything above MED_CAP is "huge")
    uint64_t run = 0;
    for (uint32_t base = 0; base < c; base += MED_THREADS) {
      const uint32_t i = base + tid;
      const uint64_t li = i < c ? a.src_len[beg + i] : 0u;
      uint64_t tot;
      const uint64_t ex = block_exclusive_scan(li, s_ws, tot);
      if (i < c) s_moff[i] = (uint32_t)min(run + ex, (uint64_t)MED_CAP + 1);
      run += tot;
    }
    if (run > MED_CAP) {  // uniform
      if (tid == 0) {
        const uint32_t at = atomicAdd(a.n_huge, 1u);
        a.huge_rec[at] = rec;
        a.huge_bucket[at] = bucket;
      }
      continue;
    }
    const uint32_t L = (uint32_t)run;
    if (tid == 0) s_moff[c] = L;
    __syncthreads();
    const uint32_t outn = cta_union_term<NW>(a.src_ptr + beg, c, L, a.rem, s_v, s_o, s_moff, s_cnt, s_last);
    uint32_t* const oth = s_v;  // the survivors
    // ---- output space, then the stream and the values
    if (tid == 0) {
      s_pos[0] = atomicAdd(&a.out_cursor[0], (unsigned long long)outn);
      s_pos[1] = a.want_enc ? atomicAdd(&a.out_cursor[1], (unsigned long long)intcomp::enc_bound(outn)) : 0ull;
    }
    __syncthreads();
    uint32_t* const dst_post = a.out_post + s_pos[0];
    uint32_t* const dst_enc = a.out_enc + s_pos[1];
    for (uint32_t e = tid; e < outn; e += MED_THREADS) dst_post[e] = oth[e];
    uint32_t enc = 0;
    if (a.want_enc && outn >= 128) {
      enc = intcomp::enc_emit_cta(oth, outn, dst_enc, s_table, s_stage, s_ws);
    } else if (a.want_enc && outn) {
      if (warp_id() == 0) {
        const uint32_t e2 = intcomp::enc_emit_warp(oth, outn, dst_enc, s_stage);
        if (lane_id() == 0) s_table[0] = e2;
      }
      __syncthreads();
      enc = s_table[0];
    }
    if (tid == 0) {
      GroupRec& r = a.recs[rec];
      r.cnt = outn;
      r.enc = enc;
      r.dec = reinterpret_cast<uint64_t>(dst_post);
      r.eoff = reinterpret_cast<uint64_t>(dst_enc);
      if (outn || a.keep_empty) {
        unsigned long long* bo = reinterpret_cast<unsigned long long*>(a.bk_raw);
        atomicAdd(&bo[0ull * a.nb1 + bucket], 1ull);
        atomicAdd(&bo[1ull * a.nb1 + bucket], (unsigned long long)r.tlen);
        atomicAdd(&bo[2ull * a.nb1 + bucket], (unsigned long long)outn);
        atomicAdd(&bo[3ull * a.nb1 + bucket], (unsigned long long)enc);
      }
    }
  }
}

// ---------------------------------------------------------------- point read (one term)
// Read(min == max): the whole call as ONE kernel.  A warp per segment looks the term up (32-way
// search, one equality check) and records where its list lies; the last CTA to finish unions the
// <= k lists with cta_union_term (up to 4096 values; sorted + deduped when >= 2 segments hold the
// term, passed through for one: survey Q4), applies the removed filter and writes the one-term
// result and its counts — to the result arrays and to pinned host memory.  The general path
// (windows, plan, bucket kernel, totals, placement: five dependent kernels, ~75 us) remains for
// anything larger; status 2 tells the host to take it.
constexpr uint32_t kPointCap = 8 * MED_RUN;  // 4096 values
enum : uint32_t { kPointAbsent = 0xFFFFFFFFu };
struct PointArgs {
  const SegDesc* segs;     // pinned host table (tb / toff / post / poff / n)
  int k;
  const uint8_t* term;     // pinned host
  uint32_t tlen;
  RemovedSet rem;
  int keep_empty;
  uint64_t* src_ptr;       // [2 k] scratch: by segment, then compacted
  uint32_t* src_len;       // [k]
  uint8_t* o_term_bytes;
  uint32_t* o_term_off;    // [2]
  uint32_t* o_post;        // [kPointCap]
  uint64_t* o_post_off;    // [2]
  uint64_t* h_res;         // pinned: status (1 done, 2 too large), T, P, postings in, sources
  uint32_t* ticket;
};

__global__ void __launch_bounds__(256) k4_point_kernel(const PointArgs a) {
  pdl_enter();
  __shared__ uint32_t s_v[kPointCap];
  __shared__ uint32_t s_o[kPointCap + kPointCap / 16];
  __shared__ uint32_t s_moff[kMaxSegs + 1];
  __shared__ uint64_t s_ws[256 / 32 + 2];
  __shared__ uint32_t s_ws32[256 / 32 + 2];
  __shared__ uint32_t s_cnt[8], s_last[8];
  __shared__ bool s_is_last;
  const uint32_t tid = threadIdx.x;
  const unsigned lane = lane_id(), w = warp_id();
  // the term: staged from the pinned block once per CTA
  uint8_t* const s_term = reinterpret_cast<uint8_t*>(s_o);
  const int s = blockIdx.x * 8 + (int)w;
  SegDesc sd = {};
  if (s < a.k) sd = a.segs[s];  // (requested before the term: two reads over the bus at once)
  for (uint32_t i = tid; i < a.tlen; i += 256) s_term[i] = a.term[i];
  __syncthreads();
  if (s < a.k) {
    auto term_vs = [&](uint32_t i) {
      const uint32_t o = __ldg(sd.toff + i), n = __ldg(sd.toff + i + 1) - o;
      return term_compare(sd.tb + o, n, s_term, a.tlen);
    };
    const uint32_t lo = warp_partition_point(0u, sd.n, [&](uint32_t i) { return term_vs(i) < 0; });
    const bool found = lo < sd.n && term_vs(lo) == 0;
    if (lane == 0) {
      uint64_t ptr = 0;
      uint32_t len = kPointAbsent;
      if (found) {
        const uint64_t p0 = __ldg(sd.poff + lo), p1 = __ldg(sd.poff + lo + 1);
        ptr = reinterpret_cast<uint64_t>(sd.post + p0);
        len = (uint32_t)min(p1 - p0, (uint64_t)kPointCap + 1);
      }
      a.src_ptr[s] = ptr;
      a.src_len[s] = len;
    }
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) s_is_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_is_last) return;
  __threadfence();
  // ---- the last CTA: the segments that hold the term, in segment order
  uint64_t* const cptr = a.src_ptr + a.k;
  uint32_t c = 0;
  uint64_t L = 0;
  for (int base = 0; base < a.k; base += 256) {
    const int x = base + (int)tid;
    const uint32_t len = x < a.k ? *(volatile uint32_t*)(a.src_len + x) : kPointAbsent;
    const bool present = len != kPointAbsent;
    uint32_t ctot;
    uint64_t ltot;
    const uint32_t ex_c = block_exclusive_scan<uint32_t>(present ? 1u : 0u, s_ws32, ctot);
    const uint64_t ex_l = block_exclusive_scan<uint64_t>(present ? (uint64_t)len : 0ull, s_ws, ltot);
    if (present) {
      cptr[c + ex_c] = *(volatile uint64_t*)(a.src_ptr + x);
      s_moff[c + ex_c] = (uint32_t)min(L + ex_l, (uint64_t)kPointCap + 1);
    }
    c += ctot;
    L += ltot;
  }
  if (tid == 0) s_moff[c] = (uint32_t)min(L, (uint64_t)kPointCap + 1);
  __syncthreads();
  if (c == 0 || L > kPointCap) {  // uniform
    if (tid == 0) {
      a.o_term_off[0] = 0;
      a.o_post_off[0] = 0;
      a.h_res[1] = 0;
      a.h_res[2] = 0;
      a.h_res[3] = L;
      a.h_res[4] = c;
      a.h_res[0] = c == 0 ? 1 : 2;
      *a.ticket = 0;
    }
    return;
  }
  const uint32_t outn = cta_union_term<8>(cptr, c, (uint32_t)L, a.rem, s_v, s_o, s_moff, s_cnt, s_last);
  const uint32_t T = (outn || a.keep_empty) ? 1u : 0u;
  for (uint32_t e = tid; e < outn; e += 256) a.o_post[e] = s_v[e];
  if (T)
    for (uint32_t i = tid; i < a.tlen; i += 256) a.o_term_bytes[i] = a.term[i];
  if (tid == 0) {
    a.o_term_off[0] = 0;
    a.o_term_off[1] = a.tlen;
    a.o_post_off[0] = 0;
    a.o_post_off[1] = outn;
    a.h_res[1] = T;
    a.h_res[2] = T ? outn : 0;
    a.h_res[3] = L;
    a.h_res[4] = c;
    a.h_res[0] = 1;
    *a.ticket = 0;
  }
}

int k4_point_read(const SegDesc* h_segs, int k, const uint8_t* term, uint32_t tlen,
                  const RemovedSet& rem, bool keep_empty, EmitOut& out, uint64_t* h_res,
                  cudaStream_t s) {
  if (k < 1 || k > kMaxSegs || tlen > kPointMaxTerm) return II2_ERR_INVALID;
  DevBuf<uint64_t> ptrs;
  DevBuf<uint32_t> lens;
  II2_TRY(ptrs.alloc_scratch(2 * (size_t)k, s));
  II2_TRY(lens.alloc_scratch((size_t)k, s));
  II2_TRY(out.term_bytes.alloc(tlen, s, 32));
  II2_TRY(out.term_off.alloc(2, s, 16));
  II2_TRY(out.post.alloc(kPointCap, s, 16));
  II2_TRY(out.post_off.alloc(2, s, 16));
  uint32_t* const tickets = device_tickets();
  if (!tickets) return II2_ERR_NOMEM;
  PointArgs a;
  a.segs = h_segs;
  a.k = k;
  a.term = term;
  a.tlen = tlen;
  a.rem = rem;
  a.keep_empty = keep_empty ? 1 : 0;
  a.src_ptr = ptrs.p;
  a.src_len = lens.p;
  a.o_term_bytes = out.term_bytes.p;
  a.o_term_off = out.term_off.p;
  a.o_post = out.post.p;
  a.o_post_off = out.post_off.p;
  a.h_res = h_res;
  a.ticket = tickets + 2;
  h_res[0] = 0;
  ProfScope scope("k4_point", s);
  II2_LAUNCH_CHAIN(k4_point_kernel, div_up(k, 8), 256, 0, s, a);
  return II2_OK;
}

// ---------------------------------------------------------------- heavy terms (global memory)
__global__ void __launch_bounds__(256) k2_large_len(const LargeArgs a, uint32_t n) {
  const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (g >= n) return;
  const GroupIn gi = a.gin[a.rec[g]];
  uint64_t L = 0;
  for (uint32_t j = lane_id(); j < gi.c; j += 32) L += a.src_len[gi.src + j];
  L = warp_sum(L);
  if (lane_id() == 0) a.len[g] = L;
}

__global__ void __launch_bounds__(256)
k2_large_counts(const LargeArgs a, uint32_t n, uint32_t* __restrict__ c) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n) c[g] = a.gin[a.rec[g]].c;
}

// gather: grid (x = CTAs per group, y = group)
// bitmap != null: instead of copying, set the bit of every value (bitmap path of group g0)
__global__ void __launch_bounds__(256)
k2_large_gather(const LargeArgs a, uint32_t* __restrict__ bitmap, uint32_t g0) {
  __shared__ uint64_t s_moff[kMaxSegs + 1];
  __shared__ uint64_t s_ws[256 / 32 + 2];
  const uint32_t g = bitmap ? g0 : blockIdx.y;
  if (!bitmap && a.presorted && a.presorted[g]) return;  // set straight from the sources
  const uint32_t c = a.gin[a.rec[g]].c, beg = a.gin[a.rec[g]].src;
  uint64_t run = 0;
  for (uint32_t base = 0; base < c; base += 256) {
    const uint32_t i = base + threadIdx.x;
    const uint64_t li = i < c ? a.src_len[beg + i] : 0u;
    uint64_t tot;
    const uint64_t ex = block_exclusive_scan(li, s_ws, tot);
    if (i < c) s_moff[i] = run + ex;
    run += tot;
  }
  if (threadIdx.x == 0) s_moff[c] = run;
  __syncthreads();
  const uint64_t n = run;
  uint32_t* dst = a.tmp + a.off[g];
  for (uint64_t e = (uint64_t)blockIdx.x * 256 + threadIdx.x; e < n; e += (uint64_t)gridDim.x * 256) {
    uint32_t lo = 0, hi = c;
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (s_moff[mid + 1] <= e)
        lo = mid + 1;
      else
        hi = mid;
    }
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.src_ptr[beg + lo]);
    const uint32_t x = __ldg(src + (e - s_moff[lo]));
    if (bitmap)
      atomicOr(&bitmap[x >> 5], 1u << (x & 31u));
    else
      dst[e] = x;
  }
}

constexpr uint32_t LG_TILE = 4096;

// sort every aligned LG_TILE tile of every heavy group in shared memory
__global__ void __launch_bounds__(512) k2_large_tile_sort(const LargeArgs a) {
  __shared__ uint32_t tile[LG_TILE];
  if (a.gin[a.rec[blockIdx.y]].c == 1 && !a.always_sort) return;  // single source: passes through unsorted (Q4)
  if (a.presorted && a.presorted[blockIdx.y]) return;
  const uint64_t n = a.len[blockIdx.y];
  uint32_t* base = a.tmp + a.off[blockIdx.y];
  for (uint64_t t0 = (uint64_t)blockIdx.x * LG_TILE; t0 < n; t0 += (uint64_t)gridDim.x * LG_TILE) {
    const uint32_t m = (uint32_t)((n - t0) < LG_TILE ? (n - t0) : LG_TILE);
    for (uint32_t i = threadIdx.x; i < m; i += 512) tile[i] = base[t0 + i];
    __syncthreads();
    bitonic_sort_any(tile, m, threadIdx.x, 512u, [](uint32_t x, uint32_t y) { return x < y; },
                     [] { __syncthreads(); });
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < m; i += 512) base[t0 + i] = tile[i];
    __syncthreads();
  }
}

// one global stage of the direction-free bitonic network: flip (kk, j == 0) or half-cleaner j
__global__ void __launch_bounds__(256) k2_large_stage(const LargeArgs a, uint64_t kk, uint64_t j) {
  const uint64_t n = a.len[blockIdx.y];
  if ((kk >> 1) >= n || (a.gin[a.rec[blockIdx.y]].c == 1 && !a.always_sort)) return;  // sorted / pass-through
  if (a.presorted && a.presorted[blockIdx.y]) return;
  uint32_t* v = a.tmp + a.off[blockIdx.y];
  const uint64_t half = j ? j : (kk >> 1);
  const uint64_t limit = (n + 1) / 2 + half;
  for (uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x; t < limit;
       t += (uint64_t)gridDim.x * 256) {
    uint64_t i, l;
    if (j == 0) {
      i = (t / half) * kk + (t % half);
      l = i ^ (kk - 1);
    } else {
      i = (t / j) * (j << 1) + (t % j);
      l = i + j;
    }
    if (l < n && i < n) {
      const uint32_t x = v[i], y = v[l];
      if (y < x) {
        v[i] = y;
        v[l] = x;
      }
    }
  }
}

// finish block size kk inside shared memory: half-cleaners j = LG_TILE/2 .. 1
__global__ void __launch_bounds__(512) k2_large_tile_merge(const LargeArgs a, uint64_t kk) {
  __shared__ uint32_t tile[LG_TILE];
  const uint64_t n = a.len[blockIdx.y];
  if ((kk >> 1) >= n || (a.gin[a.rec[blockIdx.y]].c == 1 && !a.always_sort)) return;
  if (a.presorted && a.presorted[blockIdx.y]) return;
  uint32_t* base = a.tmp + a.off[blockIdx.y];
  for (uint64_t t0 = (uint64_t)blockIdx.x * LG_TILE; t0 < n; t0 += (uint64_t)gridDim.x * LG_TILE) {
    const uint32_t m = (uint32_t)((n - t0) < LG_TILE ? (n - t0) : LG_TILE);
    for (uint32_t i = threadIdx.x; i < m; i += 512) tile[i] = base[t0 + i];
    __syncthreads();
    for (uint32_t j = LG_TILE / 2; j >= 1; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < LG_TILE / 2; t += 512) {
        const uint32_t i = (t / j) * (j << 1) + (t % j);
        const uint32_t l = i + j;
        if (l < m) {
          const uint32_t x = tile[i], y = tile[l];
          if (y < x) {
            tile[i] = y;
            tile[l] = x;
          }
        }
      }
      __syncthreads();
    }
    for (uint32_t i = threadIdx.x; i < m; i += 512) base[t0 + i] = tile[i];
    __syncthreads();
  }
}

// ---- very long unions over a dense id range: bitmap instead of a sort ------------------------
// A union of n values whose largest id is M costs O(n log^2 n) on the bitonic path; when M is
// not much larger than n (a stop-word term, a short prefix: most ids of the universe are hit)
// setting one bit per value in an M-bit map (L2-resident up to a few hundred MB... 2 MiB for a
// 2^24 universe) and reading the map back in order is the sorted-unique union in O(n + M/32).
constexpr uint64_t BM_MIN_VALUES = 1ull << 16;  // shorter unions stay on the sort path
constexpr uint32_t BM_CHUNK_WORDS = 32;         // one warp expands 1024 bits

__global__ void __launch_bounds__(256)
k2_bm_max(const LargeArgs a, uint32_t g, uint32_t* __restrict__ out) {
  const GroupIn gi = a.gin[a.rec[g]];
  uint32_t m = 0;
  // one warp per source at a time; the sources of a group are few and long here
  const uint32_t warps = gridDim.x * (blockDim.x >> 5);
  for (uint32_t j = blockIdx.x * (blockDim.x >> 5) + warp_id(); j < gi.c; j += warps) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.src_ptr[gi.src + j]);
    const uint32_t n = a.src_len[gi.src + j];
    for (uint32_t e = lane_id(); e < n; e += 32) m = max(m, __ldg(src + e));
  }
  m = __reduce_max_sync(0xffffffffu, m);
  if (lane_id() == 0 && m) atomicMax(out, m);
}

// counts[c] = set bits of chunk c (32 words); counts[n_chunks] = 0 for the scan
// (the removed filter is applied here, on whole words, when the removed set has its own bitmap)
__global__ void __launch_bounds__(256)
k2_bm_count(uint32_t* __restrict__ bitmap, uint64_t words, uint64_t n_chunks,
            uint64_t* __restrict__ counts, const RemovedSet rem) {
  const uint64_t c = ((uint64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  if (c > n_chunks) return;
  const uint64_t w = c * BM_CHUNK_WORDS + lane_id();
  uint32_t x = (c < n_chunks && w < words) ? bitmap[w] : 0u;
  if (x && rem.bitmap && (w << 5) < rem.bitmap_bits) {  // bitmap_bits is a multiple of 32
    x &= ~__ldg(rem.bitmap + w);
    bitmap[w] = x;
  }
  const uint32_t tot = __reduce_add_sync(0xffffffffu, __popc(x));
  if (lane_id() == 0) counts[c] = tot;
}

// the set bits of chunk c, ascending, to out[pos[c] ...); the last warp records the total
__global__ void __launch_bounds__(256)
k2_bm_expand(const uint32_t* __restrict__ bitmap, uint64_t words, uint64_t n_chunks,
             const uint64_t* __restrict__ pos, uint32_t* __restrict__ out,
             uint64_t* __restrict__ len_out) {
  const uint64_t c = ((uint64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  if (c >= n_chunks) return;
  const unsigned lane = lane_id();
  const uint64_t w = c * BM_CHUNK_WORDS + lane;
  uint32_t x = w < words ? bitmap[w] : 0u;
  const uint32_t cnt = __popc(x);
  const uint32_t inc = warp_inclusive_scan(cnt);
  uint32_t* dst = out + pos[c] + (inc - cnt);
  const uint32_t base = (uint32_t)(w << 5);
  while (x) {
    const uint32_t b = __ffs(x) - 1;
    x &= x - 1;
    *dst++ = base + b;
  }
  if (c + 1 == n_chunks && lane == 31) *len_out = pos[c] + inc;
}

// one CTA per heavy group: in-place dedup + filter, encode, record, bucket totals
__global__ void __launch_bounds__(1024) k2_large_finish(const LargeArgs a) {
  __shared__ uint64_t s_ws[1024 / 32 + 2];
  __shared__ uint32_t s_stage[32 * intcomp::kStageWords];
  __shared__ uint32_t s_enc;
  const uint32_t g = blockIdx.x;
  const uint64_t n = a.len[g];
  const bool single = a.gin[a.rec[g]].c == 1 && !a.always_sort;  // pass-through: duplicates stay
  uint32_t* v = a.tmp + a.off[g];
  uint64_t outn = 0;
  // bitmap path: already sorted, deduped and (when the removed set has a bitmap) filtered
  const bool done = a.presorted && a.presorted[g] && (a.rem.n == 0 || a.rem.bitmap != nullptr);
  if (done) outn = n;
  for (uint64_t e0 = 0; e0 < n && !done; e0 += 1024) {
    const uint64_t e = e0 + threadIdx.x;
    const bool valid = e < n;
    const uint32_t x = valid ? v[e] : 0u;
    const uint64_t keep =
        (valid && (single || e == 0 || v[e - 1] != x) && !is_removed(a.rem, x)) ? 1u : 0u;
    uint64_t tot;
    const uint64_t ex = block_exclusive_scan(keep, s_ws, tot);  // syncs: reads precede writes
    if (keep) v[outn + ex] = x;
    outn += tot;
    __syncthreads();
  }
  __threadfence_block();
  __syncthreads();
  uint32_t* enc_dst = a.enc + a.eoff[g];
  if (a.want_enc && outn >= 4096) {
    // all 32 warps: block sizes -> prefix -> blocks in parallel.  The slot holds
    // n + n/4 + 8 words; its last outn/128 words are free while the stream is written
    // (the stream ends before them for every list of >= 670 values) and hold the block table.
    uint32_t* table = enc_dst + (n + n / 4 + 8) - (outn >> 7);
    const uint32_t enc = intcomp::enc_emit_cta(v, (uint32_t)outn, enc_dst, table, s_stage, s_ws);
    if (threadIdx.x == 0) s_enc = enc;
  } else if (warp_id() == 0) {
    uint32_t enc = 0;
    if (a.want_enc && outn) enc = intcomp::enc_emit_warp(v, (uint32_t)outn, enc_dst, s_stage);
    if (lane_id() == 0) s_enc = enc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    GroupRec& r = a.recs[a.rec[g]];
    r.cnt = (uint32_t)outn;
    r.enc = s_enc;
    r.dec = reinterpret_cast<uint64_t>(v);
    r.eoff = reinterpret_cast<uint64_t>(a.enc + a.eoff[g]);
    if (a.bk_raw && (outn || a.keep_empty)) {
      const uint32_t b = a.bucket[g];
      unsigned long long* bo = reinterpret_cast<unsigned long long*>(a.bk_raw);
      atomicAdd(&bo[0ull * a.nb1 + b], 1ull);
      atomicAdd(&bo[1ull * a.nb1 + b], (unsigned long long)r.tlen);
      atomicAdd(&bo[2ull * a.nb1 + b], (unsigned long long)outn);
      atomicAdd(&bo[3ull * a.nb1 + b], (unsigned long long)s_enc);
    }
  }
}

// The multi-CTA union of `h_nl` heavy groups (also the per-prefix union of k5_prefix.cu).  The
// caller fills rec / bucket / gin / src_ptr / src_len / recs / rem / flags / bk_raw; sizes,
// offsets and the sort space are set up here.  Synchronises the stream.
int k2_large_run(LargeArgs la, uint32_t h_nl, DevBuf<uint32_t>& large_tmp,
                 DevBuf<uint32_t>& large_enc, cudaStream_t s) {
  if (h_nl == 0) return II2_OK;
  const bool want_enc = la.want_enc != 0;
  DevBuf<uint64_t> d_len, d_off;
  II2_TRY(d_len.alloc_scratch(h_nl, s));
  II2_TRY(d_off.alloc_scratch(2 * (size_t)h_nl, s));
  la.len = d_len.p;
  la.off = d_off.p;
  la.eoff = d_off.p + h_nl;
  la.tmp = nullptr;
  la.enc = nullptr;
  k2_large_len<<<div_up((uint64_t)h_nl * 32, 256), 256, 0, s>>>(la, h_nl);
  II2_LAUNCHED();
  std::vector<uint64_t> lens(h_nl), offs(2 * (size_t)h_nl);
  II2_CUDA_TRY(cudaMemcpyAsync(lens.data(), d_len.p, (size_t)h_nl * 8, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  uint64_t total = 0, etotal = 0;
  for (uint32_t i = 0; i < h_nl; i++) {
    if (lens[i] >= (1ull << 32)) {
      set_last_error("a single term unions %llu postings (max 2^32-1)",
                     (unsigned long long)lens[i]);
      return II2_ERR_UNSUPPORTED;
    }
    offs[i] = total;
    offs[h_nl + i] = etotal;
    total += lens[i];
    etotal += lens[i] + lens[i] / 4 + 8;
  }
  II2_TRY(large_tmp.alloc_scratch(total, s));
  if (want_enc) II2_TRY(large_enc.alloc_scratch(etotal, s));
  la.tmp = large_tmp.p;
  la.enc = large_enc.p;
  // which groups take the bitmap path: long, sortable, and dense enough (map words <= 4 n)
  std::vector<uint8_t> h_pre(h_nl, 0);
  std::vector<uint32_t> h_max(h_nl, 0);
  DevBuf<uint8_t> d_pre;
  DevBuf<uint32_t> d_max, bm_words;
  DevBuf<uint64_t> bm_counts;
  la.presorted = nullptr;
  {
    std::vector<uint32_t> cand;
    for (uint32_t i = 0; i < h_nl; i++)
      if (lens[i] >= BM_MIN_VALUES) cand.push_back(i);
    if (!cand.empty()) {
      std::vector<uint32_t> h_c(h_nl);
      II2_TRY(d_max.alloc_scratch(h_nl, s));
      II2_CUDA_TRY(cudaMemsetAsync(d_max.p, 0, (size_t)h_nl * 4, s));
      for (uint32_t i : cand) {
        k2_bm_max<<<148, 256, 0, s>>>(la, i, d_max.p + i);
        II2_LAUNCHED();
      }
      II2_CUDA_TRY(cudaMemcpyAsync(h_max.data(), d_max.p, (size_t)h_nl * 4, cudaMemcpyDeviceToHost, s));
      // single-source groups pass through unsorted unless always_sort: read their source counts
      DevBuf<uint32_t> d_c;
      II2_TRY(d_c.alloc_scratch(h_nl, s));
      k2_large_counts<<<div_up(h_nl, 256), 256, 0, s>>>(la, h_nl, d_c.p);
      II2_LAUNCHED();
      II2_CUDA_TRY(cudaMemcpyAsync(h_c.data(), d_c.p, (size_t)h_nl * 4, cudaMemcpyDeviceToHost, s));
      II2_CUDA_TRY(cudaStreamSynchronize(s));
      uint64_t max_words = 0;
      bool any = false;
      for (uint32_t i : cand) {
        const uint64_t words = ((uint64_t)h_max[i] >> 5) + 1;
        if ((h_c[i] > 1 || la.always_sort) && words <= 4 * lens[i]) {
          h_pre[i] = 1;
          any = true;
          max_words = std::max(max_words, words);
        }
      }
      if (any) {
        II2_TRY(d_pre.alloc_scratch(h_nl, s));
        II2_CUDA_TRY(cudaMemcpyAsync(d_pre.p, h_pre.data(), h_nl, cudaMemcpyHostToDevice, s));
        II2_TRY(bm_words.alloc_scratch(max_words + BM_CHUNK_WORDS, s));
        II2_TRY(bm_counts.alloc_scratch((max_words + BM_CHUNK_WORDS - 1) / BM_CHUNK_WORDS + 2, s));
        la.presorted = d_pre.p;
      }
    }
  }
  II2_CUDA_TRY(cudaMemcpyAsync(d_off.p, offs.data(), 2 * (size_t)h_nl * 8, cudaMemcpyHostToDevice, s));
  for (uint32_t y0 = 0; y0 < h_nl; y0 += 32768) {  // grid.y limit
    const uint32_t ny = std::min<uint32_t>(32768, h_nl - y0);
    uint64_t maxL = 0;
    for (uint32_t i = 0; i < ny; i++) maxL = std::max(maxL, lens[y0 + i]);
    LargeArgs b2 = la;
    b2.rec += y0;
    if (b2.presorted) b2.presorted += y0;
    if (b2.bucket) b2.bucket += y0;
    b2.len += y0;
    b2.off += y0;
    b2.eoff += y0;
    const unsigned gx = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((maxL + 4095) / 4096, 2048));
    dim3 grid(gx, ny);
    k2_large_gather<<<grid, 256, 0, s>>>(b2, nullptr, 0);
    II2_LAUNCHED();
    // dense long unions: bitmap path, one group after the other (they are few)
    uint64_t maxS = 0;  // longest union left to the sort path
    for (uint32_t i = 0; i < ny; i++) {
      const uint32_t g = y0 + i;
      if (!h_pre[g]) {
        maxS = std::max(maxS, lens[g]);
        continue;
      }
      const uint64_t words = ((uint64_t)h_max[g] >> 5) + 1;
      const uint64_t n_chunks = (words + BM_CHUNK_WORDS - 1) / BM_CHUNK_WORDS;
      II2_CUDA_TRY(cudaMemsetAsync(bm_words.p, 0, words * 4, s));
      k2_large_gather<<<(unsigned)std::min<uint64_t>((lens[g] + 255) / 256, 148 * 16), 256, 0, s>>>(
          b2, bm_words.p, i);
      II2_LAUNCHED();
      k2_bm_count<<<div_up((n_chunks + 1) * 32, 256), 256, 0, s>>>(bm_words.p, words, n_chunks,
                                                                   bm_counts.p, la.rem);
      II2_LAUNCHED();
      II2_TRY(exclusive_scan_u64(bm_counts.p, n_chunks + 1, nullptr, s));
      k2_bm_expand<<<div_up(n_chunks * 32, 256), 256, 0, s>>>(bm_words.p, words, n_chunks,
                                                              bm_counts.p, la.tmp + offs[g],
                                                              d_len.p + g);
      II2_LAUNCHED();
    }
    maxL = maxS;
    k2_large_tile_sort<<<grid, 512, 0, s>>>(b2);
    II2_LAUNCHED();
    for (uint64_t kk = 2ull * LG_TILE; (kk >> 1) < maxL; kk <<= 1) {
      k2_large_stage<<<grid, 256, 0, s>>>(b2, kk, 0);
      II2_LAUNCHED();
      for (uint64_t j = kk >> 2; j >= LG_TILE; j >>= 1) {
        k2_large_stage<<<grid, 256, 0, s>>>(b2, kk, j);
        II2_LAUNCHED();
      }
      k2_large_tile_merge<<<grid, 512, 0, s>>>(b2, kk);
      II2_LAUNCHED();
    }
    k2_large_finish<<<ny, 1024, 0, s>>>(b2);
    II2_LAUNCHED();
  }
  II2_CUDA_TRY(cudaStreamSynchronize(s));  // keeps `offs` alive until its copy is done
  return II2_OK;
}

// ---------------------------------------------------------------- host driver
// Does a call of N instances over k segments take the fused bucket kernel?
static bool k12_takes_fused(uint64_t N, int k) {
  const char* fused_env = getenv("II2_FUSED");
  const bool fused_on = fused_env ? atoi(fused_env) != 0 : N <= 65536;
  return fused_on && k12f_supported(k);
}

int k12_union(const MergePlan& plan, const RemovedSet& rem, bool want_dec, bool want_enc,
              bool keep_empty, uint64_t n_in, uint64_t tb_in, UnionOut& u, cudaStream_t s) {
  u.keep_empty = keep_empty;
  u.want_dec = want_dec;
  u.want_enc = want_enc;
  const uint32_t B = plan.n_buckets, N = plan.n_total;
  const int k = plan.k;
  // II2_FUSED=1: the one-kernel-per-bucket path (k12_fused.cu) with the general kernels for the
  // buckets it passes.  Measured on B200 (profiles/r02_experiments.md): 2.3 ms for 86 % of the C2
  // instances + 0.46 ms for the rest against 2.3 ms for K1b + K2b over all of them, so the
  // general kernels stay the default; the fused path moves 1.6x fewer DRAM bytes per step.
  // Small calls (narrow range reads) are launch-latency bound and the fused path has three
  // launches fewer: 185 vs 219 us for a 0.1 % read of C3; it takes them unless II2_FUSED=0.
  u.fused = k12_takes_fused(N, k);
  DevBuf<GroupIn> gin;
  DevBuf<uint64_t> src_ptr;
  DevBuf<uint32_t> src_len;
  II2_TRY(gin.alloc_scratch(N, s));
  II2_TRY(src_ptr.alloc_scratch(N, s));
  II2_TRY(src_len.alloc_scratch(N, s));
  II2_TRY(u.recs.alloc_scratch(N, s));
  II2_TRY(u.bk_D.alloc_scratch(B, s));
  II2_TRY(u.bk_raw.alloc_scratch(4 * (size_t)(B + 1), s));
  II2_TRY(u.bk_out.alloc_scratch(4 * (size_t)(B + 1), s));
  // totals[0..3] scan totals, [4] terms merged, [6] n_large (u32), [7] deferred buckets (u32)
  II2_TRY(u.totals.alloc_scratch(8, s));
  // `_val` staging: every light term of L values owns a slot of L + L/4 + 6 words; the bucket
  // bases are the plan's upper-bound prefix, so nothing has to be read back before K2b
  const uint64_t enc_cap = n_in + n_in / 4 + 6ull * N + 64;
  if (want_enc) II2_TRY(u.tmp_enc.alloc_scratch(enc_cap, s, 16));
  // gather slots of the light terms (K1b -> K2b); the decoded union replaces them in place
  II2_TRY(u.tmp_post.alloc_scratch(n_in, s, 16));
  const uint32_t large_cap = (uint32_t)std::min<uint64_t>(N, n_in / REG_CAP + 1);
  // [8][large_cap]: K2b's list (rec, bucket), the huge list, the lists the warp kernel and the
  // four-warp CTA kernel pass on
  DevBuf<uint32_t> large_u32;
  II2_TRY(large_u32.alloc_scratch(8 * (size_t)large_cap, s));
  // mid / medium terms (k2_mwarp_kernel, k2_medium_kernel): unions and streams bump-allocated
  // [0] postings, [1] words, [2] work cursors (2 x u32: eight-warp CTA kernel, warp kernel),
  // [3] terms passed on (2 x u32: by the warp kernel, by the four-warp CTA kernel),
  // [4] work cursor of the four-warp CTA kernel
  DevBuf<unsigned long long> med_cursor;
  II2_TRY(med_cursor.alloc_scratch(8, s));
  II2_CUDA_TRY(cudaMemsetAsync(med_cursor.p, 0, 64, s));
  II2_TRY(u.med_post.alloc_scratch(n_in, s, 16));
  if (want_enc) II2_TRY(u.med_enc.alloc_scratch(n_in + n_in / 4 + 16ull * large_cap + 64, s, 16));
  II2_CUDA_TRY(cudaMemsetAsync(u.totals.p, 0, 64, s));
  II2_CUDA_TRY(cudaMemsetAsync(u.bk_raw.p, 0, 4 * (size_t)(B + 1) * 8, s));
  II2_TRY(u.bk_mode.alloc_scratch(B, s));
  if (u.fused) {
    II2_TRY(u.st_tb.alloc_scratch(tb_in, s, 64));
    II2_TRY(u.st_off.alloc_scratch(3 * (size_t)N, s));
    II2_TRY(u.def_list.alloc_scratch(B, s));
  } else {
    II2_CUDA_TRY(cudaMemsetAsync(u.bk_mode.p, 0, (size_t)B * 4, s));  // K12F_RECORDS
  }

  K1bArgs a1;
  a1.segs = plan.segs;
  a1.k = k;
  a1.part = plan.part.p;
  a1.btb = plan.btb.p;
  a1.bpo = plan.bpo.p;
  a1.bk_pos = plan.bk_pos();
  a1.bk_cpl = plan.bk_cpl.p;
  a1.bk_P = plan.bk_P();
  a1.gin = gin.p;
  a1.gath = u.tmp_post.p;
  a1.src_ptr = src_ptr.p;
  a1.src_len = src_len.p;
  a1.bk_D = u.bk_D.p;
  K2bArgs a2;
  a2.bk_pos = plan.bk_pos();
  a2.bk_P = plan.bk_P();
  a2.bk_E = plan.bk_E();
  a2.bk_D = u.bk_D.p;
  a2.gin = gin.p;
  a2.rem = rem;
  a2.want_enc = want_enc ? 1 : 0;
  a2.want_dec = want_dec ? 1 : 0;
  a2.keep_empty = keep_empty ? 1 : 0;
  a2.recs = u.recs.p;
  a2.gath = u.tmp_post.p;
  a2.tmp_enc = u.tmp_enc.p;
  a2.bk_raw = u.bk_raw.p;
  a2.nb1 = B + 1;
  a2.n_large = reinterpret_cast<uint32_t*>(u.totals.p + 6);
  a2.large_rec = large_u32.p;
  a2.large_bucket = large_u32.p + large_cap;
  const size_t smem = k1b_smem_bytes(k);
  static size_t attr = 0;
  if (smem > attr) {
    const size_t want = std::max(k1b_smem_bytes(kMaxSegs), smem);
    II2_CUDA_TRY(cudaFuncSetAttribute(k1b_group_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)want));
    II2_CUDA_TRY(cudaFuncSetAttribute(k1b_group_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)want));
    attr = want;
  }
  // the general kernels over `grid` buckets: all of them, or the list K12f deferred
  auto general = [&](uint32_t grid, const uint32_t* list) -> int {
    a1.bucket0 = a2.bucket0 = 0;
    a1.list = a2.list = list;
    {
      ProfScope scope("k1b_group", s);
      if (list) {
        II2_LAUNCH_CHAIN(k1b_group_kernel<true>, grid, K1B_THREADS, smem, s, a1);
      } else {
        II2_LAUNCH_CHAIN(k1b_group_kernel<false>, grid, K1B_THREADS, smem, s, a1);
      }
    }
    {
      ProfScope scope("k2b_union", s);
      if (list) {
        II2_LAUNCH_CHAIN(k2b_union_kernel<true>, grid, K2B_THREADS, 0, s, a2);
      } else {
        II2_LAUNCH_CHAIN(k2b_union_kernel<false>, grid, K2B_THREADS, 0, s, a2);
      }
    }
    {  // the terms K2b deferred: up to MW_CAP values one warp each, up to 4096 one CTA each;
       // device-side work lists, no host round trip
      ProfScope scope("k2_medium", s);
      uint32_t* const mid_rec = large_u32.p + 4 * (size_t)large_cap;
      uint32_t* const mid_bucket = large_u32.p + 5 * (size_t)large_cap;
      uint32_t* const n_mid = reinterpret_cast<uint32_t*>(med_cursor.p + 3);
      MwArgs w2;
      w2.n_in_list = a2.n_large;
      w2.in_rec = a2.large_rec;
      w2.in_bucket = a2.large_bucket;
      w2.gin = gin.p;
      w2.src_ptr = src_ptr.p;
      w2.src_len = src_len.p;
      w2.recs = u.recs.p;
      w2.rem = rem;
      w2.want_enc = want_enc ? 1 : 0;
      w2.keep_empty = keep_empty ? 1 : 0;
      w2.bk_raw = u.bk_raw.p;
      w2.nb1 = B + 1;
      w2.cursor = reinterpret_cast<uint32_t*>(med_cursor.p + 2) + 1;
      w2.n_out_list = n_mid;
      w2.out_rec = mid_rec;
      w2.out_bucket = mid_bucket;
      w2.out_post = u.med_post.p;
      w2.out_enc = u.med_enc.p;
      w2.out_cursor = med_cursor.p;
      II2_LAUNCH_CHAIN(k2_mwarp_kernel, kNumSMs * MW_MIN_CTAS, MW_WARPS * 32, 0, s, w2);
      // one CTA per term: four warps up to 2048 values (eight CTAs per SM), eight warps up to
      // 4096 (five per SM); each passes the longer terms on through its own list
      uint32_t* const mid2_rec = large_u32.p + 6 * (size_t)large_cap;
      uint32_t* const mid2_bucket = large_u32.p + 7 * (size_t)large_cap;
      uint32_t* const n_mid2 = reinterpret_cast<uint32_t*>(med_cursor.p + 3) + 1;
      MedArgs m;
      m.n_large = n_mid;
      m.large_rec = mid_rec;
      m.large_bucket = mid_bucket;
      m.gin = gin.p;
      m.src_ptr = src_ptr.p;
      m.src_len = src_len.p;
      m.recs = u.recs.p;
      m.rem = rem;
      m.want_enc = want_enc ? 1 : 0;
      m.keep_empty = keep_empty ? 1 : 0;
      m.bk_raw = u.bk_raw.p;
      m.nb1 = B + 1;
      m.cursor = reinterpret_cast<uint32_t*>(med_cursor.p + 4);
      m.n_huge = n_mid2;
      m.huge_rec = mid2_rec;
      m.huge_bucket = mid2_bucket;
      m.out_post = u.med_post.p;
      m.out_enc = u.med_enc.p;
      m.out_cursor = med_cursor.p;
      II2_LAUNCH_CHAIN(k2_medium_kernel<4>, kNumSMs * 8, 4 * 32, 0, s, m);
      m.n_large = n_mid2;
      m.large_rec = mid2_rec;
      m.large_bucket = mid2_bucket;
      m.cursor = reinterpret_cast<uint32_t*>(med_cursor.p + 2);
      m.n_huge = a2.n_large + 1;  // the high half of totals[6]
      m.huge_rec = large_u32.p + 2 * (size_t)large_cap;
      m.huge_bucket = large_u32.p + 3 * (size_t)large_cap;
      II2_LAUNCH_CHAIN(k2_medium_kernel<8>, kNumSMs * 5, 8 * 32, 0, s, m);
    }
    return II2_OK;
  };
  uint64_t* h_tot = pinned_scratch();  // 8 words
  if (!h_tot) return II2_ERR_NOMEM;
  // bucket totals -> prefixes -> host (synchronises the stream)
  auto totals = [&](bool emit_early = false) -> int {
    ProfScope scope("k12_scan_sync", s);
    // four scans, Σ bk_D (terms_merged) and the copy of the eight totals to the host: one launch
    II2_TRY(exclusive_scan_multi_sum_to_host(u.bk_raw.p, u.bk_out.p, B + 1, 4, u.totals.p, u.bk_D.p, B,
                                             4, h_tot, 8, s));
    if (emit_early) II2_TRY(k6_emit_early(plan, u, n_in, tb_in, *u.early_out, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    return II2_OK;
  };
  if (u.fused) {
    K12fArgs f;
    f.segs = plan.segs;
    f.k = k;
    f.part = plan.part.p;
    f.btb = plan.btb.p;
    f.bpo = plan.bpo.p;
    f.bk_pos = plan.bk_pos();
    f.bk_cpl = plan.bk_cpl.p;
    f.bk_P = plan.bk_P();
    f.bk_E = plan.bk_E();
    f.bk_TB = plan.bk_TB();
    f.rem = rem;
    f.want_enc = want_enc ? 1 : 0;
    f.want_dec = want_dec ? 1 : 0;
    f.keep_empty = keep_empty ? 1 : 0;
    f.bk_D = u.bk_D.p;
    f.bk_mode = u.bk_mode.p;
    f.bk_raw = u.bk_raw.p;
    f.nb1 = B + 1;
    f.st_tb = u.st_tb.p;
    f.st_toff = u.st_off.p;
    f.st_eoff = u.st_off.p + N;
    f.st_poff = u.st_off.p + 2 * (size_t)N;
    f.st_enc = u.tmp_enc.p;
    f.st_post = u.tmp_post.p;
    f.n_def = reinterpret_cast<uint32_t*>(u.totals.p + 7);
    f.def_list = u.def_list.p;
    {
      ProfScope scope("k12f_bucket", s);
      II2_TRY(k12f_launch(f, B, s));
    }
    // optimistic: scan right away (and, for a small call, place the result before waiting);
    // redone only if buckets were deferred
    II2_TRY(totals(u.early_out != nullptr));
    u.n_def = (uint32_t)h_tot[7];
    if (u.n_def) {
      II2_TRY(general(u.n_def, u.def_list.p));
      II2_TRY(totals());
    }
  } else {
    // (running the two kernels chunk-wise on two streams was measured slower on B200 than back
    // to back: 3.27 vs 2.94 ms)
    II2_TRY(general(B, nullptr));
    II2_TRY(totals());
  }
  const uint32_t h_nl = (uint32_t)(h_tot[6] >> 32);  // terms the CTA kernels passed on (> 4096 values)
  if (h_nl > 0) {
    ProfScope scope("k2_large", s);
    LargeArgs la;
    la.rec = large_u32.p + 2 * (size_t)large_cap;
    la.bucket = large_u32.p + 3 * (size_t)large_cap;
    la.gin = gin.p;
    la.src_ptr = src_ptr.p;
    la.src_len = src_len.p;
    la.recs = u.recs.p;
    la.rem = rem;
    la.want_enc = want_enc ? 1 : 0;
    la.keep_empty = keep_empty ? 1 : 0;
    la.always_sort = 0;
    la.presorted = nullptr;
    la.bk_raw = u.bk_raw.p;
    la.nb1 = B + 1;
    II2_TRY(k2_large_run(la, h_nl, u.large_tmp, u.large_enc, s));
    II2_TRY(totals());
  }
  for (int i = 0; i < 4; i++) u.h_totals[i] = h_tot[i];
  u.terms_merged = h_tot[4];
  return II2_OK;
}

}  // namespace ii2
