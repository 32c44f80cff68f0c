// union_dev.cuh — device building blocks shared by the union kernels (K2b in k12_union.cu, the
// fused bucket kernel in k12_fused.cu): the blocked register sorting network, the per-term
// union + dedup + removed filter (file.MergeTermValues file/types.go:14-22, filter
// shard.go:181-190) and the shared-memory intcomp encoders (intcomp.CompressUint32,
// file/writer.go:49).
#pragma once
#include "intcomp.cuh"
#include "union.cuh"

namespace ii2 {

constexpr uint32_t REG_CAP = 256;  // values a warp sorts in registers

// staging words that certainly hold the intcomp stream of n values (oracle/intcomp_ref.c
// orc_intcomp_bound: 3 + 129 per block + 1 + ceil(5 * tail / 4) + 1; at most two blocks here)
__host__ __device__ __forceinline__ uint32_t enc_slot_words(uint32_t n) { return n + (n >> 2) + 6; }

// ---- union of one term by a group of W lanes (W = 16: two terms per warp; W = 32: one) ------
// The term's values live BLOCKED in registers: lane hl of the group holds elements
// hl*8 .. hl*8+7.  Eight values per lane keep most compare-exchanges of the sorting network
// inside a thread (two min/max instructions, no shuffle): a local 19-comparator network sorts
// the eight, then one bitonic merge level per doubling — a mirrored "flip" across lanes, the
// half-cleaners whose distance is a whole number of lanes (one shuffle + one predicated
// min/max per value), and three local half-cleaners (distance 4, 2, 1).  The shuffle pipe
// and shared memory share one data path on the SM and were the busiest unit of the striped
// version (ncu: lsu wavefronts 66 %), hence this layout: 80 shuffles sort two 128-value terms.
__device__ __forceinline__ void cex(uint32_t& x, uint32_t& y) {
  const uint32_t lo = min(x, y), hi = max(x, y);
  x = lo;
  y = hi;
}

__device__ __forceinline__ void sort8_local(uint32_t (&v)[8]) {
  cex(v[0], v[1]); cex(v[2], v[3]); cex(v[4], v[5]); cex(v[6], v[7]);
  cex(v[0], v[2]); cex(v[1], v[3]); cex(v[4], v[6]); cex(v[5], v[7]);
  cex(v[1], v[2]); cex(v[5], v[6]); cex(v[0], v[4]); cex(v[3], v[7]);
  cex(v[1], v[5]); cex(v[2], v[6]);
  cex(v[1], v[4]); cex(v[3], v[6]);
  cex(v[2], v[4]); cex(v[3], v[5]);
  cex(v[3], v[4]);
}

__device__ __forceinline__ void clean8_local(uint32_t (&v)[8]) {
  cex(v[0], v[4]); cex(v[1], v[5]); cex(v[2], v[6]); cex(v[3], v[7]);
  cex(v[0], v[2]); cex(v[1], v[3]); cex(v[4], v[6]); cex(v[5], v[7]);
  cex(v[0], v[1]); cex(v[2], v[3]); cex(v[4], v[5]); cex(v[6], v[7]);
}

// one merge level: blocks of K elements (K/8 lanes) become sorted; K >= 16
template <int K>
__device__ __forceinline__ void merge_level(uint32_t (&v)[8], unsigned hl) {
  {  // flip: element e pairs with e ^ (K-1) = (lane ^ (K/8-1), 7 - r)
    const bool lower = (hl & (K / 16)) == 0;
    uint32_t o[8];
#pragma unroll
    for (int r = 0; r < 8; r++) o[r] = __shfl_xor_sync(0xffffffffu, v[7 - r], K / 8 - 1);
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = lower ? min(v[r], o[r]) : max(v[r], o[r]);
  }
#pragma unroll
  for (int j = K / 4; j >= 8; j >>= 1) {  // half-cleaners across lanes
    const bool lower = (hl & (j / 8)) == 0;
#pragma unroll
    for (int r = 0; r < 8; r++) {
      const uint32_t o = __shfl_xor_sync(0xffffffffu, v[r], j / 8);
      v[r] = lower ? min(v[r], o) : max(v[r], o);
    }
  }
  clean8_local(v);
}

// sorts the 8*W values of every group; nmax = largest real length in the warp (padding is
// 0xFFFFFFFF at the end, so levels whose blocks would only hold padding are skipped)
template <int W>
__device__ __forceinline__ void sort_blocked(uint32_t (&v)[8], unsigned hl, uint32_t nmax) {
  sort8_local(v);
  if (nmax > 8) merge_level<16>(v, hl);
  if (nmax > 16) merge_level<32>(v, hl);
  if (nmax > 32) merge_level<64>(v, hl);
  if (nmax > 64) merge_level<128>(v, hl);
  if (W == 32 && nmax > 128) merge_level<256>(v, hl);
}

// ---- the same network with V values per lane over a whole warp (V * 32 values) ----------------
// Used for terms of REG_CAP < L <= 1024 values (k12_union.cu, k2_mwarp_kernel): 32 values per
// lane keep five of every six compare-exchanges of a 1024-value sort inside a thread.
template <int V>
__device__ __forceinline__ void sort_local_v(uint32_t (&v)[V]) {  // bitonic network, ascending
#pragma unroll
  for (int k = 2; k <= V; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
      for (int i = 0; i < V; i++) {
        const int l = i ^ j;
        if (l > i) {
          const uint32_t lo = min(v[i], v[l]), hi = max(v[i], v[l]);
          const bool asc = (i & k) == 0;  // compile time
          v[i] = asc ? lo : hi;
          v[l] = asc ? hi : lo;
        }
      }
    }
  }
}

template <int V>
__device__ __forceinline__ void clean_local_v(uint32_t (&v)[V]) {  // bitonic -> ascending
#pragma unroll
  for (int d = V / 2; d > 0; d >>= 1) {
#pragma unroll
    for (int i = 0; i < V; i++)
      if ((i & d) == 0) cex(v[i], v[i + d]);
  }
}

// Sorts the V * 32 values of the warp; n = real length (padding 0xFFFFFFFF at the end).  The
// merge levels are ONE rolled loop over the block size K (the shuffle distance is a run-time
// value): fully unrolled, five levels of a 32-values-per-lane network are ~35 KB of SASS and the
// kernel starved on instruction fetch (ncu: `no_inst` the top stall of every min / max).
// Level K: blocks of K elements (K / V lanes) become sorted —
//   flip: element e pairs with e ^ (K-1) = (lane ^ (K/V - 1), V-1-r), two values at a time;
//   half-cleaners whose distance is a whole number of lanes; then the local half-cleaners.
template <int V>
__device__ __forceinline__ void sort_warp_v(uint32_t (&v)[V], unsigned lane, uint32_t n) {
  sort_local_v<V>(v);
#pragma unroll 1
  for (uint32_t K = 2 * V; K <= 32 * V && n > K / 2; K <<= 1) {
    {
      const unsigned dist = K / V - 1;
      const bool lower = (lane & (K / (2 * V))) == 0;
#pragma unroll
      for (int r = 0; r < V / 2; r++) {
        const uint32_t a = v[r], b = v[V - 1 - r];
        const uint32_t oa = __shfl_xor_sync(0xffffffffu, b, dist);
        const uint32_t ob = __shfl_xor_sync(0xffffffffu, a, dist);
        v[r] = ((a < oa) == lower) ? a : oa;
        v[V - 1 - r] = ((b < ob) == lower) ? b : ob;
      }
    }
#pragma unroll 1
    for (uint32_t j = K / 4; j >= V; j >>= 1) {
      const unsigned dist = j / V;
      const bool lower = (lane & dist) == 0;
#pragma unroll
      for (int r = 0; r < V; r++) {
        const uint32_t o = __shfl_xor_sync(0xffffffffu, v[r], dist);
        v[r] = ((v[r] < o) == lower) ? v[r] : o;
      }
    }
    clean_local_v<V>(v);
  }
}

// The part of a merge level that stays inside a warp once the cross-warp stages are done
// (k12_union.cu, k2_medium_kernel): half-cleaners at lane distances 16 .. 1, then the local ones.
template <int V>
__device__ __forceinline__ void clean_warp_v(uint32_t (&v)[V], unsigned lane) {
#pragma unroll 1
  for (unsigned dist = 16; dist >= 1; dist >>= 1) {
    const bool lower = (lane & dist) == 0;
#pragma unroll
    for (int r = 0; r < V; r++) {
      const uint32_t o = __shfl_xor_sync(0xffffffffu, v[r], dist);
      v[r] = ((v[r] < o) == lower) ? v[r] : o;
    }
  }
  clean_local_v<V>(v);
}

// Union of the term of this lane's group: L gathered values at `slot` (global) -> sorted
// (slices.Sort) and deduped (slices.Compact) when the term has >= 2 sources (a single-source
// term passes through in source order, duplicates kept: survey Q4) -> removed filter ->
// survivors compacted into buf[0..outn) (shared, this group's).  Every lane of the warp must
// call; groups with nothing to do pass L = 0.  Returns outn (uniform inside the group).
template <int W>
__device__ __forceinline__ uint32_t union_blocked(const uint32_t* slot, uint32_t* buf, uint32_t L,
                                                  bool multi, const RemovedSet& rem) {
  const unsigned lane = lane_id(), hl = lane & (W - 1);
  uint32_t v[8];
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const uint32_t e = hl * 8 + r;
    v[r] = e < L ? slot[e] : 0xFFFFFFFFu;
  }
  const bool any_multi = __any_sync(0xffffffffu, multi && L > 1);
  if (any_multi) {
    const uint32_t nmax = __reduce_max_sync(0xffffffffu, multi ? L : 0u);
    sort_blocked<W>(v, hl, nmax);
    if (!multi) {  // the other group of the warp holds a pass-through term: undo
#pragma unroll
      for (int r = 0; r < 8; r++) {
        const uint32_t e = hl * 8 + r;
        v[r] = e < L ? slot[e] : 0xFFFFFFFFu;
      }
    }
  }
  // all membership probes first: eight independent loads in flight per lane
  uint32_t keep = 0;
  if (rem.bitmap) {  // bit v of the bitmap <=> v removed, for v < bitmap_bits (<= 2^29)
    const uint32_t nbits = (uint32_t)rem.bitmap_bits;
    uint32_t word[8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
      const bool probe = hl * 8 + r < L && v[r] < nbits;
      word[r] = probe ? __ldg(rem.bitmap + (v[r] >> 5)) : 0u;
    }
#pragma unroll
    for (int r = 0; r < 8; r++)
      keep |= (hl * 8 + r < L && !((word[r] >> (v[r] & 31u)) & 1u)) ? 1u << r : 0u;
  } else {
#pragma unroll
    for (int r = 0; r < 8; r++)
      if (hl * 8 + r < L && !is_removed(rem, v[r])) keep |= 1u << r;
  }
  const uint32_t up = __shfl_up_sync(0xffffffffu, v[7], 1, W);  // last value of the lane below
  if (multi) {  // drop a value equal to its predecessor (sorted order)
    if (hl > 0 && up == v[0]) keep &= ~1u;
#pragma unroll
    for (int r = 1; r < 8; r++)
      if (v[r] == v[r - 1]) keep &= ~(1u << r);
  }
  const uint32_t cnt = __popc(keep);
  uint32_t inc = cnt;
#pragma unroll
  for (int d = 1; d < W; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d, W);
    if (hl >= (unsigned)d) inc += o;
  }
  const uint32_t outn = __shfl_sync(0xffffffffu, inc, W - 1, W);
  uint32_t* dst = buf + (inc - cnt);
#pragma unroll
  for (int r = 0; r < 8; r++) {  // predicated store + pointer bump: no branches
    const bool k = (keep >> r) & 1u;
    if (k) *dst = v[r];
    dst += k ? 1 : 0;
  }
  __syncwarp();
  return outn;
}

// intcomp.CompressUint32 of v[0..n), n <= 127 (one var-byte section: count word, then
// zigzag deltas, 7 bits per byte, low group first, last byte |= 0x80, first delta against 0;
// oracle/intcomp_ref.c), by a group of W lanes: lane hl codes values hl*8 .. hl*8+7.
// v and out are the group's shared buffers (16-byte aligned).  Returns the words (uniform in
// the group); n = 0 -> 0.  Every lane of the warp must call.
template <int W>
__device__ __forceinline__ uint32_t encode_small_blocked(const uint32_t* v, uint32_t n,
                                                         uint32_t* out) {
  const unsigned hl = lane_id() & (W - 1);
  const uint32_t e0 = hl * 8;
  // values past n read as garbage inside the group's buffer and get length 0
  const uint4 a = *reinterpret_cast<const uint4*>(v + e0);
  const uint4 b = *reinterpret_cast<const uint4*>(v + e0 + 4);
  const uint32_t x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  uint32_t prev = e0 ? v[e0 - 1] : 0u;
  uint32_t z[8], lens = 0, bytes = 0;  // lens: 4 bits per value
#pragma unroll
  for (int r = 0; r < 8; r++) {
    z[r] = intcomp::zigzag(x[r], prev);
    prev = x[r];
    // ceil(bitlen / 7) for bitlen in 1..32 (z = 0 codes as one byte): (bitlen + 6) * 37 >> 8
    const uint32_t bl = 32u - __clz(z[r] | 1u);
    const uint32_t len = e0 + r < n ? ((bl + 6u) * 37u) >> 8 : 0u;
    lens |= len << (4 * r);
    bytes += len;
  }
  uint32_t inc = bytes;
#pragma unroll
  for (int d = 1; d < W; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d, W);
    if (hl >= (unsigned)d) inc += o;
  }
  const uint32_t total = __shfl_sync(0xffffffffu, inc, W - 1, W);
  // byte stores predicated in PTX: the compiler would chain branches (len > 1 implies
  // len > 0 ...), five of them per value
  uint32_t sb = (uint32_t)__cvta_generic_to_shared(out + 1) + (inc - bytes);
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const uint32_t zz = z[r];
    const uint32_t len = (lens >> (4 * r)) & 15u;
    // the low four 7-bit groups spread over four bytes, terminator bit on the last byte
    uint32_t w = (zz & 0x7Fu) | ((zz << 1) & 0x7F00u) | ((zz << 2) & 0x7F0000u) |
                 ((zz << 3) & 0x7F000000u);
    const uint32_t term = 0x80u << ((8 * len - 8) & 31u);
    w |= len <= 4 ? term : 0u;  // (len 0 stores nothing)
    const uint32_t b4 = (zz >> 28) | 0x80u;
    asm volatile(
        "{\n\t"
        ".reg .pred p0, p1, p2, p3, p4;\n\t"
        ".reg .b32 t1, t2, t3;\n\t"
        "setp.gt.u32 p0, %1, 0;\n\t"
        "setp.gt.u32 p1, %1, 1;\n\t"
        "setp.gt.u32 p2, %1, 2;\n\t"
        "setp.gt.u32 p3, %1, 3;\n\t"
        "setp.gt.u32 p4, %1, 4;\n\t"
        "shr.u32 t1, %2, 8;\n\t"
        "shr.u32 t2, %2, 16;\n\t"
        "shr.u32 t3, %2, 24;\n\t"
        "@p0 st.shared.u8 [%0], %2;\n\t"
        "@p1 st.shared.u8 [%0+1], t1;\n\t"
        "@p2 st.shared.u8 [%0+2], t2;\n\t"
        "@p3 st.shared.u8 [%0+3], t3;\n\t"
        "@p4 st.shared.u8 [%0+4], %3;\n\t"
        "}"
        :
        : "r"(sb), "r"(len), "r"(w), "r"(b4)
        : "memory");
    sb += len;
  }
  if (n) {
    if (hl == 0) out[0] = n;
    uint8_t* end = reinterpret_cast<uint8_t*>(out + 1) + total;
    if (hl < ((4u - (total & 3u)) & 3u)) end[hl] = 0;  // zero padding of the last word
  }
  __syncwarp();  // no lane leaves early: the groups of a warp meet here
  return n ? 1 + (total + 3) / 4 : 0u;
}

// intcomp.CompressUint32 of v[0..n) (shared memory) into out (shared memory, a different
// buffer, at least enc_bound(n) words), one pass with rolled loops.  Returns the stream
// length in words (uniform).
__device__ __forceinline__ uint32_t encode_shared_warp(const uint32_t* v, uint32_t n, uint32_t* out) {
  if (n == 0) return 0;
  const unsigned lane = lane_id();
  const uint32_t nb = n >> 7, tail = n & 127u;
  uint32_t pos = 0;
  if (nb) {
    pos = 3;
#pragma unroll 1
    for (uint32_t blk = 0; blk < nb; blk++) {
      const uint32_t hpos = pos++;
      uint32_t hdr = 0;
#pragma unroll 1
      for (uint32_t g = 0; g < 4; g++) {
        const uint32_t idx = blk * 128 + g * 32 + lane;
        const uint32_t cur = v[idx];
        const uint32_t prev = idx ? v[idx - 1] : cur;
        const uint32_t z = intcomp::zigzag(cur, prev);
        const uint32_t m = __reduce_or_sync(0xffffffffu, z);
        const uint32_t sgn = m & 1u;
        const uint32_t bw = sgn ? intcomp::bitlen(m) : intcomp::bitlen(m >> 1);
        const uint32_t coded = sgn ? z : (cur - prev);
        hdr |= ((sgn << 7) | bw) << (24 - 8 * g);
        if (bw == 32) {
          out[pos + lane] = coded;
        } else if (bw > 0) {
          if (lane < bw) out[pos + lane] = 0;
          __syncwarp();
          const uint32_t bit = lane * bw, sh = bit & 31u;
          atomicOr(&out[pos + (bit >> 5)], coded << sh);
          if (sh + bw > 32u) atomicOr(&out[pos + (bit >> 5) + 1], coded >> (32u - sh));
        }
        pos += bw;
      }
      if (lane == 0) out[hpos] = hdr;
    }
    if (lane == 0) {
      out[0] = nb * 128;
      out[1] = pos;
      out[2] = v[0];
    }
  }
  if (tail) {
    if (lane == 0) out[pos] = tail;
    pos += 1;
    uint8_t* sb = reinterpret_cast<uint8_t*>(out + pos);
    uint32_t bo = 0;
#pragma unroll 1
    for (uint32_t t0 = 0; t0 < tail; t0 += 32) {
      const uint32_t i = t0 + lane;
      uint32_t z = 0, len = 0;
      if (i < tail) {
        const uint32_t idx = nb * 128 + i;
        z = intcomp::zigzag(v[idx], i ? v[idx - 1] : 0u);
        len = intcomp::vbyte_len(z);
      }
      const uint32_t inc = warp_inclusive_scan(len);
      const uint32_t off = bo + inc - len;
      // 7 bits per byte, low group first, the last byte carries 0x80
      if (len > 0) sb[off] = (uint8_t)((z & 0x7Fu) | (len == 1 ? 0x80u : 0u));
      if (len > 1) sb[off + 1] = (uint8_t)(((z >> 7) & 0x7Fu) | (len == 2 ? 0x80u : 0u));
      if (len > 2) sb[off + 2] = (uint8_t)(((z >> 14) & 0x7Fu) | (len == 3 ? 0x80u : 0u));
      if (len > 3) sb[off + 3] = (uint8_t)(((z >> 21) & 0x7Fu) | (len == 4 ? 0x80u : 0u));
      if (len > 4) sb[off + 4] = (uint8_t)(((z >> 28) & 0x7Fu) | 0x80u);
      bo += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane < ((4u - (bo & 3u)) & 3u)) sb[bo + lane] = 0;  // zero padding of the last word
    pos += (bo + 3) / 4;
  }
  __syncwarp();
  return pos;
}

// ---- union of one term by a whole CTA (k2_medium_kernel, the point read, the batched lookup) ----
constexpr int MED_V = 16;                 // values per lane of a warp-sorted run
constexpr uint32_t MED_RUN = 32 * MED_V;  // 512
// Word of s_o that holds gathered value e: runs of MED_RUN values, one pad word per 16.
__device__ __forceinline__ uint32_t med_run_slot(uint32_t e) { return e + (e >> 4); }

// The union of ONE term by a CTA of NW warps (k2_medium_kernel, api.cu's point read): c sources
// (g_ptr[0 .. c), lengths as the prefix s_moff[0 .. c], L = s_moff[c] <= NW * 512 values) are
// gathered into shared memory, sorted and deduped when c >= 2 (a single source passes through in
// its own order, duplicates kept: survey Q4), filtered against the removed set and compacted.
// Every thread of the CTA calls; returns the number of survivors, which end in s_v[0 .. outn).
// s_v: NW * 512 words, s_o: NW * 512 * 17 / 16 words, s_cnt / s_last: NW words.
template <int NW>
__device__ __forceinline__ uint32_t cta_union_term(const uint64_t* __restrict__ g_ptr, uint32_t c,
                                                   uint32_t L, const RemovedSet& rem, uint32_t* s_v,
                                                   uint32_t* s_o, const uint32_t* s_moff,
                                                   uint32_t* s_cnt, uint32_t* s_last) {
  constexpr int MED_THREADS = NW * 32;
  const uint32_t tid = threadIdx.x;
  // ---- gather.  The term lands in s_o as runs of MED_RUN values (one per warp), every run
  // padded (one word per 16) so that the blocked register load below is free of bank
  // conflicts; the tail up to a power-of-two number of runs is the sentinel 0xFFFFFFFF.
  const bool single = c == 1;  // passes through unsorted, duplicates kept (survey Q4)
  const uint32_t w = warp_id(), lane = lane_id();
  uint32_t nrun = 1;
  while (nrun * MED_RUN < L) nrun <<= 1;
  const uint32_t Lpad = nrun * MED_RUN;
  // The source pointers wait in s_v (free until the first exchange) and every thread resolves
  // eight elements before it stores any: eight value loads in flight instead of a chain of
  // pointer load -> value load per element.
  uint64_t* const s_ptr = reinterpret_cast<uint64_t*>(s_v);
  const uint32_t* const src0 = reinterpret_cast<const uint32_t*>(g_ptr[0]);
  if (!single) {
    for (uint32_t i = tid; i < c; i += MED_THREADS) s_ptr[i] = g_ptr[i];
    __syncthreads();
  }
  uint32_t top = 1;  // largest power of two below c
  while (top * 2 < c) top <<= 1;
  const bool by_source = !single && c * 8 <= L;  // sources of >= 8 values on average
  if (by_source) {
    // a warp per source, two sources (eight loads per lane) in flight; no search at all
    for (uint32_t e = L + tid; e < Lpad; e += MED_THREADS) s_o[med_run_slot(e)] = 0xFFFFFFFFu;
    for (uint32_t j0 = 2 * w; j0 < c; j0 += 2 * (MED_THREADS / 32)) {
      uint32_t x[2][4], o2[2], n2[2];
      const uint32_t* p2[2];
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const uint32_t j = j0 + q;
        const bool in = j < c;
        p2[q] = reinterpret_cast<const uint32_t*>(in ? s_ptr[j] : 0ull);
        o2[q] = in ? s_moff[j] : 0u;
        n2[q] = in ? s_moff[j + 1] - o2[q] : 0u;
#pragma unroll
        for (int t = 0; t < 4; t++) x[q][t] = t * 32 + lane < n2[q] ? __ldg(p2[q] + t * 32 + lane) : 0u;
      }
#pragma unroll
      for (int q = 0; q < 2; q++) {
#pragma unroll
        for (int t = 0; t < 4; t++)
          if (t * 32 + lane < n2[q]) s_o[med_run_slot(o2[q] + t * 32 + lane)] = x[q][t];
        for (uint32_t i = 128 + lane; i < n2[q]; i += 32) s_o[med_run_slot(o2[q] + i)] = __ldg(p2[q] + i);
      }
    }
  }
  for (uint32_t e0 = tid; e0 < (by_source ? 0u : Lpad); e0 += 8 * MED_THREADS) {
    uint32_t x[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const uint32_t e = e0 + q * MED_THREADS;
      x[q] = 0xFFFFFFFFu;
      if (e < L) {
        if (single) {
          x[q] = __ldg(src0 + e);
        } else {
          uint32_t lo = 0;  // last source whose first element is <= e (empty sources skipped)
          for (uint32_t st = top; st; st >>= 1) {
            const uint32_t m = lo + st;
            if (m < c && s_moff[m] <= e) lo = m;
          }
          x[q] = __ldg(reinterpret_cast<const uint32_t*>(s_ptr[lo]) + (e - s_moff[lo]));
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const uint32_t e = e0 + q * MED_THREADS;
      if (e < Lpad) s_o[med_run_slot(e)] = x[q];
    }
  }
  __syncthreads();
  // ---- sort.  From here to the compaction the values live in registers: warp w holds run w,
  // lane l its values 16 l .. 16 l + 15.  Each run is sorted by its warp (sort_warp_v<16>);
  // then 1 / 2 / 3 bitonic merge levels double the sorted blocks up to Lpad.  A level starts
  // with the stages whose partner sits in another warp — the flip (value e against the
  // mirrored value of the partner run), then half-cleaners at warp distances — exchanged
  // through shared memory in a transposed, conflict-free layout, alternating between the two
  // buffers so that one barrier per stage is enough; the rest of the level is shuffles and
  // register compare-exchanges (clean_warp_v).
  const bool active = w < nrun;
  uint32_t v[MED_V];
#pragma unroll
  for (int r = 0; r < MED_V; r++)
    v[r] = active ? s_o[med_run_slot(w * MED_RUN + lane * MED_V + r)] : 0xFFFFFFFFu;
  if (!single) {
    {
      const uint32_t at = w * MED_RUN, n = L > at ? min(L - at, MED_RUN) : 0u;
      if (n > 1) sort_warp_v<MED_V>(v, lane, n);
    }
    uint32_t stage = 0;
    for (uint32_t nw = 2; nw <= nrun; nw <<= 1) {  // warps per sorted block after this level
      for (uint32_t dw = nw; dw >= 2; dw >>= 1) {  // dw == nw: the flip; below: half-cleaners
        const bool flip = dw == nw;
        uint32_t* const X = (stage++ & 1u) ? s_o : s_v;
        if (active) {
#pragma unroll
          for (int r = 0; r < MED_V; r++) X[w * MED_RUN + r * 32 + lane] = v[r];
        }
        __syncthreads();
        if (active) {
          const uint32_t pw = flip ? (w ^ (nw - 1)) : (w ^ (dw >> 1));
          const bool lower = (w & (dw >> 1)) == 0;
          const uint32_t* const P = X + pw * MED_RUN;
#pragma unroll
          for (int r = 0; r < MED_V; r++) {
            const uint32_t o = flip ? P[(MED_V - 1 - r) * 32 + (31 - lane)] : P[r * 32 + lane];
            v[r] = ((v[r] < o) == lower) ? v[r] : o;
          }
        }
      }
      if (active) clean_warp_v<MED_V>(v, lane);
    }
  }
  // ---- dedup + removed filter + compaction, still from the registers: sixteen membership
  // probes per lane issued eight at a time, keep flags in a register, positions from one warp
  // scan + the warps' totals; the survivors end in s_v.
  uint32_t outn;
  {
    if (lane == 31) s_last[w] = v[MED_V - 1];
    __syncthreads();  // (also: every partner has read the last exchange buffer)
    const uint32_t e_l = w * MED_RUN + lane * MED_V;  // index of v[0]
    uint32_t keep = 0;
    if (rem.bitmap) {
      const uint32_t nbits = (uint32_t)rem.bitmap_bits;
#pragma unroll
      for (int r0 = 0; r0 < MED_V; r0 += 8) {
        uint32_t word[8];
#pragma unroll
        for (int r = 0; r < 8; r++) {
          const bool probe = e_l + r0 + r < L && v[r0 + r] < nbits;
          word[r] = probe ? __ldg(rem.bitmap + (v[r0 + r] >> 5)) : 0u;
        }
#pragma unroll
        for (int r = 0; r < 8; r++)
          keep |= (e_l + r0 + r < L && !((word[r] >> (v[r0 + r] & 31u)) & 1u)) ? 1u << (r0 + r) : 0u;
      }
    } else {
#pragma unroll
      for (int r = 0; r < MED_V; r++)
        if (e_l + r < L && !(rem.n && is_removed_call(rem.sorted, rem.n, v[r]))) keep |= 1u << r;
    }
    uint32_t up = __shfl_up_sync(0xffffffffu, v[MED_V - 1], 1);  // the value before v[0]
    if (lane == 0 && w > 0) up = s_last[w - 1];
    if (!single) {
      if (e_l > 0 && up == v[0]) keep &= ~1u;
#pragma unroll
      for (int r = 1; r < MED_V; r++)
        if (v[r] == v[r - 1]) keep &= ~(1u << r);
    }
    const uint32_t cnt = __popc(keep);
    const uint32_t inc = warp_inclusive_scan(cnt);
    if (lane == 31) s_cnt[w] = inc;
    __syncthreads();
    uint32_t at = inc - cnt, tot = 0;
#pragma unroll
    for (int q = 0; q < MED_THREADS / 32; q++) {
      const uint32_t cq = s_cnt[q];
      at += (uint32_t)q < w ? cq : 0u;
      tot += cq;
    }
    outn = tot;
    uint32_t* dst = s_v + at;
#pragma unroll
    for (int r = 0; r < MED_V; r++) {
      const bool k = (keep >> r) & 1u;
      if (k) *dst = v[r];
      dst += k ? 1 : 0;
    }
  }
  __syncthreads();
  return outn;
}

}  // namespace ii2
