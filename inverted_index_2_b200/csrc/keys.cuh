// keys.cuh — fixed-width comparison keys for variable-length terms.
//
// Ordering contract = Go bytes.Compare (file/types.go:24-26): unsigned lexicographic, a proper
// prefix sorts first.  A 16-byte big-endian window (zero padded past the end of the term)
// followed by the length reproduces it for every pair of terms that share the bytes before the
// window: equal windows mean the shorter term is a prefix of the longer one unless BOTH run
// past the window, in which case the tails decide.
#pragma once
#include "common.cuh"

namespace ii2 {

// Bytes [c, c+16) of the term at tb+g0 (length len >= c) as two big-endian u64, zero padded
// past the end.  Five aligned 32-bit loads + funnel shifts (three aligned 64-bit loads were
// measured equal and would need 8-byte alignment); tb must be 4-byte aligned and readable 24
// bytes past the last term byte (segment term buffers are padded by 32).
__device__ __forceinline__ void load_key16(const uint8_t* __restrict__ tb, uint32_t g0,
                                           uint32_t len, uint32_t c, uint64_t& hi, uint64_t& lo) {
  const uint32_t avail = len - c;
  if (avail == 0) {
    hi = lo = 0;
    return;
  }
  const uint32_t a = g0 + c;
  const uint32_t* wp = reinterpret_cast<const uint32_t*>(tb + (a & ~3u));
  const uint32_t sh = (a & 3u) * 8u;
  uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2), w3 = __ldg(wp + 3),
           w4 = __ldg(wp + 4);
  uint32_t x0 = __byte_perm(__funnelshift_r(w0, w1, sh), 0, 0x0123);
  uint32_t x1 = __byte_perm(__funnelshift_r(w1, w2, sh), 0, 0x0123);
  uint32_t x2 = __byte_perm(__funnelshift_r(w2, w3, sh), 0, 0x0123);
  uint32_t x3 = __byte_perm(__funnelshift_r(w3, w4, sh), 0, 0x0123);
  hi = ((uint64_t)x0 << 32) | x1;
  lo = ((uint64_t)x2 << 32) | x3;
  if (avail < 16) {
    if (avail <= 8) {
      lo = 0;
      if (avail < 8) hi &= ~0ull << (8 * (8 - avail));
    } else {
      lo &= ~0ull << (8 * (16 - avail));
    }
  }
}

// Bytes [c+16, c+24) of the term as one big-endian u64, zero padded past the end (0 when the
// term ends inside the 16-byte window).  Same alignment / padding contract as load_key16
// (the allocation must be readable 32 bytes past the last term byte).
__device__ __forceinline__ uint64_t load_key_x(const uint8_t* __restrict__ tb, uint32_t g0,
                                               uint32_t len, uint32_t c) {
  if (len <= c + 16) return 0;
  const uint32_t avail = len - c - 16;
  const uint32_t a = g0 + c + 16;
  const uint32_t* wp = reinterpret_cast<const uint32_t*>(tb + (a & ~3u));
  const uint32_t sh = (a & 3u) * 8u;
  const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
  const uint32_t x0 = __byte_perm(__funnelshift_r(w0, w1, sh), 0, 0x0123);
  const uint32_t x1 = __byte_perm(__funnelshift_r(w1, w2, sh), 0, 0x0123);
  uint64_t x = ((uint64_t)x0 << 32) | x1;
  if (avail < 8) x &= ~0ull << (8 * (8 - avail));
  return x;
}

// A term with its leading 16-byte window cached.
struct KeyedTerm {
  uint64_t hi, lo;
  const uint8_t* p;  // first byte of the term
  uint32_t len;
};

__device__ __forceinline__ KeyedTerm keyed_term(const SegDesc& sd, uint32_t idx) {
  KeyedTerm t;
  const uint32_t o = __ldg(sd.toff + idx);
  t.len = __ldg(sd.toff + idx + 1) - o;
  t.p = sd.tb + o;
  load_key16(sd.tb, o, t.len, 0, t.hi, t.lo);
  return t;
}

// bytes.Compare(a, b) as <0, 0, >0
__device__ __forceinline__ int keyed_compare(const KeyedTerm& a, const KeyedTerm& b) {
  if (a.hi != b.hi) return a.hi < b.hi ? -1 : 1;
  if (a.lo != b.lo) return a.lo < b.lo ? -1 : 1;
  if (a.len > 16 && b.len > 16) return term_compare(a.p + 16, a.len - 16, b.p + 16, b.len - 16);
  return a.len < b.len ? -1 : (a.len > b.len ? 1 : 0);
}

// First index in [lo,hi) of segment sd whose term is >= x (vellum Iterator(min) seek).
__device__ __forceinline__ uint32_t keyed_lower_bound(const SegDesc& sd, uint32_t lo, uint32_t hi,
                                                      const KeyedTerm& x) {
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (keyed_compare(keyed_term(sd, mid), x) < 0)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

}  // namespace ii2
