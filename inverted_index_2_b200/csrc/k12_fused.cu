// k12_fused.cu — K12f: one bucket of the k-way merge from its inputs to its finished output in
// ONE kernel, everything in between in shared memory.
//
// Replaces, for one bucket of the merged term order (plan.cuh):
//   - go-iterators' MergingIterator over per-segment readers (built at shard.go:267, ordering
//     file.CompareTermValues = bytes.Compare, file/types.go:24-26) — equal terms grouped by a
//     shared-memory hash table, the distinct terms ranked;
//   - file.MergeTermValues (file/types.go:14-22), the removed filter and empty-term drop of the
//     merge loop (shard.go:181-194) and intcomp.CompressUint32 (file/writer.go:49) — the union
//     kernels of union_dev.cuh, run on a gather slot in shared memory;
//   - the reader's run-by-offsets rule (file/reader.go:50-52) — offsets, term bytes and postings
//     of the bucket's run in every segment are four contiguous pieces of that segment.
//
// Pass structure (what the split K1b -> K2b -> K6 pipeline of round 1 paid twice or three
// times): every input byte is read from HBM once — the bucket's 4 * k runs are staged with
// 16-byte asynchronous copies (cp.async.cg, LDGSTS.128) over the 16-byte aligned envelope of
// each run, the boundaries coming from the partition's tables, so there is ONE dependent round
// trip (boundary rows -> runs) instead of four (part -> offsets -> term bytes -> postings) —
// and the finished bucket (term bytes, offsets, `_val` words, decoded postings) is written once,
// densely, in merged order, to the bucket's staging area; the placement kernel (k6_emit.cu) then
// moves whole buckets with vector copies.
//
// A bucket that does not fit the fast path (more than F_CAP_I instances, runs larger than the
// staging areas, a term of more than REG_CAP values, more than F_MAXK segments) is DEFERRED: its
// number goes on a list and the general kernels of k12_union.cu (K1b / K2b / heavy-term path)
// process it afterwards.  Integer/byte work, no tensor cores.
#include "keys.cuh"
#include "union_dev.cuh"

namespace ii2 {

constexpr int F_THREADS = 512;
constexpr int F_MIN_CTAS = 2;
constexpr int F_WARPS = F_THREADS / 32;
constexpr uint32_t F_CAP_I = 1024;               // instances of a bucket
constexpr int F_PER = (F_CAP_I + F_THREADS - 1) / F_THREADS;  // instances per thread
constexpr uint32_t F_HT = F_CAP_I > 512 ? 2048 : 1024;  // hash slots (a power of two >= 2 * F_CAP_I)
constexpr uint32_t F_A_CH = F_CAP_I * 5 / 4;     // 16-byte chunks: staged term + posting offsets
constexpr uint32_t F_C_CH = F_CAP_I;             // staged postings
constexpr uint32_t F_B_CH = F_CAP_I * 9 / 8;     // staged term bytes
constexpr uint32_t F_ARENA_W = (F_A_CH + F_C_CH) * 4;  // `_val` words of a bucket (reuses A and C)
constexpr uint32_t F_GCAP = F_CAP_I * 4;         // gather slots, words (reuses the key windows)
constexpr uint32_t F_SMALL_D = 64;               // distinct terms ranked by counting
constexpr uint32_t F_EMPTY = 0xFFFFFFFFu;
static_assert(F_CAP_I <= 1024 && F_CAP_I % 64 == 0 && F_THREADS >= 128 && F_THREADS % 32 == 0 &&
              F_HT >= 2 * F_CAP_I, "tile shape");
static_assert(F_B_CH * 16 < 65536, "term positions inside the staged bytes are 16-bit");
static_assert(F_ARENA_W < (1u << 14) && F_GCAP < (1u << 13), "packed output prefixes");

// shared memory of one CTA (bytes), k segments
__host__ __device__ inline size_t k12f_smem_bytes(int k) {
  return (size_t)(F_A_CH + F_C_CH + F_B_CH) * 16 + 64  // staging (+ slack for window over-reads)
         + (size_t)F_CAP_I * 16                        // key_hi, key_lo | gather slots
         + (size_t)F_CAP_I * (4 + 4 + 8)               // cg, pbase, pfx | copy descriptors
         + (size_t)F_CAP_I * 2 * 4                     // tsm, tlen, reps, order
         + (size_t)F_HT * 4                            // hash table | ebase, rres
         + (size_t)k * 16;                             // views
}

__device__ __forceinline__ void cp_async16(uint32_t dst_shared, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_shared), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// 16-byte chunks of the aligned envelope of [p, p + bytes)
__device__ __forceinline__ uint32_t env_chunks(const void* p, uint64_t bytes) {
  const uint64_t c = ((reinterpret_cast<uintptr_t>(p) & 15u) + bytes + 15u) >> 4;
  return c > (1u << 20) ? (1u << 20) : (uint32_t)c;
}

// Bytes [c, c+16) of the term that starts at byte `t0` of the CTA's shared memory (length len
// >= c) as two big-endian u64, zero padded past the end.  Aligned 32-bit shared loads + funnel
// shifts; up to 20 bytes past the window start are read (the staging area has slack).
__device__ __forceinline__ void smem_key16_at(const uint8_t* smem, uint32_t t0, uint32_t len,
                                              uint32_t c, uint64_t& hi, uint64_t& lo) {
  const uint32_t avail = len - c;
  if (avail == 0) {
    hi = lo = 0;
    return;
  }
  const uint32_t a = t0 + c;
  const uint32_t* wp = reinterpret_cast<const uint32_t*>(smem + (a & ~3u));
  const uint32_t sh = (a & 3u) * 8u;
  const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = wp[4];
  const uint32_t x0 = __byte_perm(__funnelshift_r(w0, w1, sh), 0, 0x0123);
  const uint32_t x1 = __byte_perm(__funnelshift_r(w1, w2, sh), 0, 0x0123);
  const uint32_t x2 = __byte_perm(__funnelshift_r(w2, w3, sh), 0, 0x0123);
  const uint32_t x3 = __byte_perm(__funnelshift_r(w3, w4, sh), 0, 0x0123);
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

__global__ void __launch_bounds__(F_THREADS, F_MIN_CTAS) k12f_bucket_kernel(const K12fArgs a) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ uint64_t s_p1[8], s_p2[8];
  __shared__ uint64_t s_ws64[F_WARPS + 2];
  __shared__ uint32_t s_ws32[F_WARPS + 2];
  __shared__ uint32_t s_nreps, s_tot[2], s_bad, s_nn, s_nw;
  __shared__ uint64_t s_total;

  const int k = a.k;
  // ---- layout (byte offsets from smem) ----
  constexpr uint32_t OFF_A = 0;                         // term + posting offsets
  constexpr uint32_t OFF_C = OFF_A + F_A_CH * 16;       // postings
  constexpr uint32_t OFF_B = OFF_C + F_C_CH * 16;       // term bytes (live until the output)
  constexpr uint32_t OFF_KEYS = OFF_B + F_B_CH * 16 + 64;
  uint8_t* sp = smem + OFF_KEYS;
  uint64_t* key_hi = reinterpret_cast<uint64_t*>(sp); sp += F_CAP_I * 8;
  uint64_t* key_lo = reinterpret_cast<uint64_t*>(sp); sp += F_CAP_I * 8;
  uint32_t* const gather = reinterpret_cast<uint32_t*>(key_hi);  // once the ranking is done
  // by representative: sources << 20 | Σ source lengths (each saturated at REG_CAP + 1)
  uint32_t* cg = reinterpret_cast<uint32_t*>(sp); sp += F_CAP_I * 4;
  uint32_t* pbase = reinterpret_cast<uint32_t*>(sp); sp += F_CAP_I * 4;  // gather slot by representative
  uint64_t* pfx = reinterpret_cast<uint64_t*>(sp); sp += F_CAP_I * 8;   // output prefixes by rank
  uint16_t* tsm = reinterpret_cast<uint16_t*>(sp); sp += F_CAP_I * 2;   // term start inside area B
  uint16_t* tlen = reinterpret_cast<uint16_t*>(sp); sp += F_CAP_I * 2;
  uint16_t* reps = reinterpret_cast<uint16_t*>(sp); sp += F_CAP_I * 2;
  uint16_t* order = reinterpret_cast<uint16_t*>(sp); sp += F_CAP_I * 2;  // representative by rank
  uint32_t* table = reinterpret_cast<uint32_t*>(sp); sp += F_HT * 4;
  uint32_t* const ebase = table;            // by representative: slot in the `_val` arena
  uint32_t* const rres = table + F_CAP_I;   // by rank: values left | words << 16
  // work lists of the union phase (ranks): terms of < 128 values go two to a warp, longer ones
  // take a whole warp each.  (over pfx, which is written after the unions)
  uint16_t* const narrow_list = reinterpret_cast<uint16_t*>(pfx);
  uint16_t* const wide_list = narrow_list + F_CAP_I;
  uint32_t* v_toff = reinterpret_cast<uint32_t*>(sp); sp += k * 4;
  uint32_t* v_poff = reinterpret_cast<uint32_t*>(sp); sp += k * 4;
  uint32_t* v_tb = reinterpret_cast<uint32_t*>(sp); sp += k * 4;
  uint32_t* v_post = reinterpret_cast<uint32_t*>(sp);
  // copy descriptors of the header (dead once the copies are issued): over cg | pbase | pfx.
  // One per (segment, array): aligned source address, destination, 16-byte chunks.
  uint4* const desc = reinterpret_cast<uint4*>(cg);
  // (4 k descriptors of 16 bytes in 16 * F_CAP_I bytes: k12f_supported bounds k)
  uint16_t* const seg_of = reps;  // segment of every instance (until the grouping appends to reps)

  const uint32_t tid = threadIdx.x;
  const unsigned lane = lane_id(), warp = warp_id();
  const uint32_t b = blockIdx.x;
  const uint64_t rec_base = a.bk_pos[b];
  const uint32_t W64 = (uint32_t)min(a.bk_pos[b + 1] - rec_base, (uint64_t)0xFFFFFFFFu);
  const uint32_t W = W64;
  if (W == 0) {
    if (tid == 0) {
      a.bk_D[b] = 0;
      a.bk_mode[b] = K12F_DENSE;
    }
    return;
  }
  auto defer = [&]() {  // uniform: every thread of the CTA takes it
    if (tid == 0) {
      a.bk_mode[b] = K12F_DEFERRED;
      a.def_list[atomicAdd(a.n_def, 1u)] = b;
    }
  };
  if (W > F_CAP_I) {
    defer();
    return;
  }

  // ---------------- (0) the bucket's run in every segment; staging layout ----------------
  // Only the warps that own segments work here (k / 32 of them); thread s sizes the aligned
  // envelopes of segment s's four runs, a scan over the segments places them, and the same
  // thread writes the four copy descriptors and the views.  view = where element 0 of the
  // run would sit if the array were indexed by the instance's position in the TILE (offsets) or
  // by the global offset (term bytes, postings), in wrapping 32-bit arithmetic.
  const uint32_t nwk = ((uint32_t)k + 31u) >> 5;
  uint64_t x1 = 0, x2 = 0, inc1 = 0, inc2 = 0;  // n | cA << 32, cB | cC << 32
  uint32_t lo_i = 0, n = 0, lo_T = 0, nT = 0, nP = 0, cT = 0;
  uint64_t lo_P = 0;
  const uint8_t *pT = nullptr, *pP = nullptr, *pB = nullptr, *pC = nullptr;
  if (warp < nwk) {
    if (tid < (uint32_t)k) {
      const uint64_t r0 = (uint64_t)b * k + tid, r1 = r0 + k;
      lo_i = a.part[r0];
      n = a.part[r1] - lo_i;
      lo_T = a.btb[r0];
      nT = a.btb[r1] - lo_T;
      lo_P = a.bpo[r0];
      const uint64_t nP64 = a.bpo[r1] - lo_P;
      nP = nP64 > 0x00FFFFFFull ? 0x00FFFFFFu : (uint32_t)nP64;
      uint32_t cA = 0, cB = 0, cC = 0;
      if (n) {
        const SegDesc& sd = a.segs[tid];
        pT = reinterpret_cast<const uint8_t*>(sd.toff + lo_i);
        pP = reinterpret_cast<const uint8_t*>(sd.poff + lo_i);
        pB = sd.tb + lo_T;
        pC = reinterpret_cast<const uint8_t*>(sd.post + lo_P);
        cT = env_chunks(pT, (uint64_t)(n + 1) * 4);
        cA = cT + env_chunks(pP, (uint64_t)(n + 1) * 8);
        cB = env_chunks(pB, nT);
        cC = env_chunks(pC, (uint64_t)nP * 4);
      }
      x1 = (uint64_t)n | ((uint64_t)cA << 32);
      x2 = (uint64_t)cB | ((uint64_t)cC << 32);
    }
    inc1 = warp_inclusive_scan(x1);
    inc2 = warp_inclusive_scan(x2);
    if (lane == 31) {
      s_p1[warp] = inc1;
      s_p2[warp] = inc2;
    }
  }
  if (tid == 0) {
    s_nreps = 0;
    s_bad = 0;
    s_nn = 0;
    s_nw = 0;
  }
  __syncthreads();
  if (warp < nwk) {
    uint64_t base1 = 0, base2 = 0, tot1 = 0, tot2 = 0;
    for (uint32_t w2 = 0; w2 < nwk; w2++) {
      const uint64_t q1 = s_p1[w2], q2 = s_p2[w2];
      if (w2 < warp) {
        base1 += q1;
        base2 += q2;
      }
      tot1 += q1;
      tot2 += q2;
    }
    const bool fits = (uint32_t)(tot1 >> 32) <= F_A_CH && (uint32_t)tot2 <= F_B_CH &&
                      (uint32_t)(tot2 >> 32) <= F_C_CH;
    if (tid == 0) s_bad = fits ? 0u : 1u;
    if (fits) {
      const uint64_t e1 = base1 + inc1 - x1, e2 = base2 + inc2 - x2;
      const uint32_t rs = (uint32_t)e1;
      if (tid < (uint32_t)k) {
        uint4 d0 = make_uint4(0u, 0u, 0u, 0u), d1 = d0, d2 = d0, d3 = d0;
        if (n) {
          const uint32_t phT = (uint32_t)(reinterpret_cast<uintptr_t>(pT) & 15u),
                         phP = (uint32_t)(reinterpret_cast<uintptr_t>(pP) & 15u),
                         phB = (uint32_t)(reinterpret_cast<uintptr_t>(pB) & 15u),
                         phC = (uint32_t)(reinterpret_cast<uintptr_t>(pC) & 15u);
          const uint32_t atT = OFF_A + (uint32_t)(e1 >> 32) * 16, atP = atT + cT * 16,
                         atB = OFF_B + (uint32_t)e2 * 16, atC = OFF_C + (uint32_t)(e2 >> 32) * 16;
          const uint64_t sT = reinterpret_cast<uintptr_t>(pT) - phT, sP = reinterpret_cast<uintptr_t>(pP) - phP,
                         sB = reinterpret_cast<uintptr_t>(pB) - phB, sC = reinterpret_cast<uintptr_t>(pC) - phC;
          d0 = make_uint4((uint32_t)sT, (uint32_t)(sT >> 32), atT, cT);
          d1 = make_uint4((uint32_t)sP, (uint32_t)(sP >> 32), atP, (uint32_t)(x1 >> 32) - cT);
          d2 = make_uint4((uint32_t)sB, (uint32_t)(sB >> 32), atB, (uint32_t)x2);
          d3 = make_uint4((uint32_t)sC, (uint32_t)(sC >> 32), atC, (uint32_t)(x2 >> 32));
          v_toff[tid] = atT + phT - rs * 4;
          v_poff[tid] = atP + phP - rs * 8;
          v_tb[tid] = atB + phB - lo_T;
          v_post[tid] = atC + phC - (uint32_t)(lo_P * 4);
        }
        desc[4 * tid] = d0;
        desc[4 * tid + 1] = d1;
        desc[4 * tid + 2] = d2;
        desc[4 * tid + 3] = d3;
      }
      // segment of every instance of the tile
      if (__all_sync(0xffffffffu, n <= 32)) {
        for (uint32_t j = 0; j < n; j++) seg_of[rs + j] = (uint16_t)tid;
      } else {
        for (int sl = 0; sl < 32; sl++) {
          const uint32_t n_sl = __shfl_sync(0xffffffffu, n, sl), rs_sl = __shfl_sync(0xffffffffu, rs, sl);
          for (uint32_t j = lane; j < n_sl; j += 32) seg_of[rs_sl + j] = (uint16_t)(warp * 32 + sl);
        }
      }
    }
  }
  __syncthreads();
  if (s_bad) {  // the runs do not fit the staging areas
    defer();
    return;
  }

  // ---------------- (1) stage the runs: 16-byte asynchronous copies ----------------
  // Four lanes per descriptor walk the aligned envelope of the run; the data keeps its phase
  // modulo 16, so 32- and 64-bit elements stay aligned.
  {
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t sub = tid & 3u;
    for (uint32_t d = tid >> 2; d < 4u * (uint32_t)k; d += F_THREADS / 4) {
      const uint4 de = desc[d];
      const uint8_t* src = reinterpret_cast<const uint8_t*>((uint64_t)de.x | ((uint64_t)de.y << 32));
      for (uint32_t c = sub; c < de.w; c += 4) cp_async16(sbase + de.z + c * 16, src + c * 16);
    }
    cp_async_wait_all();
  }
  __syncthreads();  // the runs are in shared memory; the descriptors are dead

  for (uint32_t i = tid; i < F_HT / 4; i += F_THREADS)
    reinterpret_cast<uint4*>(table)[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
  for (uint32_t i = tid; i < F_CAP_I / 4; i += F_THREADS)
    reinterpret_cast<uint4*>(cg)[i] = make_uint4(0u, 0u, 0u, 0u);

  const uint32_t cpl = a.bk_cpl[b];
  // order of two terms of the bucket whose 16-byte windows are equal
  auto tail_compare = [&](uint32_t x, uint32_t y) -> int {
    const uint32_t skip = cpl + 16;
    const uint32_t nx = tlen[x], ny = tlen[y];
    if (nx > skip && ny > skip) {
      const uint8_t* px = smem + OFF_B + tsm[x] + skip;
      const uint8_t* py = smem + OFF_B + tsm[y] + skip;
      const uint32_t m = (nx < ny ? nx : ny) - skip;
      for (uint32_t i = 0; i < m; i++) {
        const int d = (int)px[i] - (int)py[i];
        if (d) return d;
      }
    }
    return nx < ny ? -1 : (nx > ny ? 1 : 0);
  };
  auto less = [&](uint16_t x, uint16_t y) -> bool {
    const uint64_t hx = key_hi[x], hy = key_hi[y];
    if (hx != hy) return hx < hy;
    const uint64_t lx = key_lo[x], ly = key_lo[y];
    if (lx != ly) return lx < ly;
    return tail_compare(x, y) < 0;
  };

  // ---------------- (2) key windows + posting runs of every instance ----------------
  uint32_t ps[F_PER];   // first posting of the thread's instances (byte offset in shared memory)
  uint32_t pl[F_PER];   // their lengths
  uint32_t og[F_PER];   // representative << 20 | where they go inside its gather slot
#pragma unroll
  for (int j = 0; j < F_PER; j++) {
    const uint32_t i = tid + j * F_THREADS;
    pl[j] = 0;
    ps[j] = 0;
    if (i < W) {
      const uint32_t s = seg_of[i];  // the run that holds instance i
      const uint32_t* to_p = reinterpret_cast<const uint32_t*>(smem + (uint32_t)(v_toff[s] + i * 4));
      const uint64_t* po_p = reinterpret_cast<const uint64_t*>(smem + (uint32_t)(v_poff[s] + i * 8));
      const uint32_t to = to_p[0], n = to_p[1] - to;
      const uint64_t pp = po_p[0], np = po_p[1] - pp;
      const uint32_t t0 = v_tb[s] + to;  // first byte of the term in shared memory
      uint64_t kh, kl;
      smem_key16_at(smem, t0, n, cpl, kh, kl);
      key_hi[i] = kh;
      key_lo[i] = kl;
      tlen[i] = (uint16_t)n;
      tsm[i] = (uint16_t)(t0 - OFF_B);
      pl[j] = np > REG_CAP ? REG_CAP + 1 : (uint32_t)np;
      ps[j] = v_post[s] + (uint32_t)pp * 4;
    }
  }
  __syncthreads();

  // ---------------- (3) group equal terms (hash table of representatives) ----------------
#pragma unroll
  for (int j = 0; j < F_PER; j++) {
    const uint32_t i = tid + j * F_THREADS;
    if (i >= W) break;
    const uint64_t kh = key_hi[i], kl = key_lo[i];
    const uint32_t tl = tlen[i];
    uint32_t h = (uint32_t)kh * 0x9E3779B1u ^ (uint32_t)(kh >> 32) * 0x85EBCA77u ^
                 (uint32_t)kl * 0xC2B2AE3Du ^ (uint32_t)(kl >> 32) * 0x27D4EB2Fu;
    h = (h ^ (h >> 15)) * 0x2C1B3C6Du + tl;
    uint32_t slot = (h ^ (h >> 13)) & (F_HT - 1);
    uint32_t rep;
    for (;;) {
      const uint32_t prev = atomicCAS(&table[slot], F_EMPTY, i);
      if (prev == F_EMPTY) {
        rep = i;
        reps[atomicAdd(&s_nreps, 1u)] = (uint16_t)i;
        break;
      }
      // (the keys of every instance were published by the barrier above)
      if (key_hi[prev] == kh && key_lo[prev] == kl && tlen[prev] == tl &&
          (tl <= cpl + 16 || tail_compare(i, prev) == 0)) {
        rep = prev;
        break;
      }
      slot = (slot + 1) & (F_HT - 1);
    }
    og[j] = (rep << 20) | (atomicAdd(&cg[rep], (1u << 20) | pl[j]) & 0xFFFFFu);
  }
  __syncthreads();
  const uint32_t D = s_nreps;

  // ---------------- (4) order the distinct terms; slots of their lists ----------------
  // rank by counting (eight lanes per term, four terms per warp) or a bitonic network; every
  // term gets a 16-byte aligned gather slot and an upper-bound slot in the `_val` arena
  if (D <= F_SMALL_D) {
    const unsigned sub = lane & 7u;
#pragma unroll 1
    for (uint32_t t0 = warp * 4; t0 < D; t0 += F_WARPS * 4) {
      const uint32_t t = t0 + (lane >> 3);
      const bool valid = t < D;
      const uint32_t me = valid ? reps[t] : 0u;
      uint32_t rank = 0, pst = 0, est = 0;
      if (valid) {
        const uint64_t mh = key_hi[me], ml = key_lo[me];
#pragma unroll 1
        for (uint32_t j = sub; j < D; j += 8) {
          const uint32_t o = reps[j];
          const uint64_t oh = key_hi[o];
          bool lt = oh < mh;
          if (oh == mh && o != me) {  // rare: the first eight bytes past the prefix agree
            const uint64_t ol = key_lo[o];
            lt = ol != ml ? ol < ml : tail_compare(o, me) < 0;
          }
          const uint32_t len = cg[o] & 0xFFFFFu;
          rank += lt ? 1u : 0u;
          pst += lt ? (len + 3u) & ~3u : 0u;
          est += lt ? enc_slot_words(len) : 0u;
        }
      }
#pragma unroll
      for (int d = 4; d > 0; d >>= 1) {
        rank += __shfl_xor_sync(0xffffffffu, rank, d);
        pst += __shfl_xor_sync(0xffffffffu, pst, d);
        est += __shfl_xor_sync(0xffffffffu, est, d);
      }
      if (valid && sub == 0) {
        const uint32_t len = cg[me] & 0xFFFFFu;
        order[rank] = (uint16_t)me;
        pbase[me] = pst;
        ebase[me] = est;
        if (len > REG_CAP) s_bad = 1;
        if (len >= 128)
          wide_list[atomicAdd(&s_nw, 1u)] = (uint16_t)rank;
        else
          narrow_list[atomicAdd(&s_nn, 1u)] = (uint16_t)rank;
        if (rank == D - 1) {
          s_tot[0] = pst + ((len + 3u) & ~3u);
          s_tot[1] = est + enc_slot_words(len);
        }
      }
    }
  } else {
    bitonic_sort_any(reps, D, tid, (uint32_t)F_THREADS, less, [] { __syncthreads(); });
    __syncthreads();
    uint32_t run_p = 0, run_e = 0;
    for (uint32_t base = 0; base < D; base += F_THREADS) {
      const uint32_t r = base + tid;
      uint32_t me = 0, li = 0, ei = 0;
      if (r < D) {
        me = reps[r];
        const uint32_t len = cg[me] & 0xFFFFFu;
        if (len > REG_CAP) s_bad = 1;
        li = (len + 3u) & ~3u;
        ei = enc_slot_words(len);
      }
      uint32_t tp, te;
      const uint32_t xp = block_exclusive_scan(li, s_ws32, tp);
      const uint32_t xe = block_exclusive_scan(ei, s_ws32, te);
      if (r < D) {
        order[r] = (uint16_t)me;
        pbase[me] = run_p + xp;
        ebase[me] = run_e + xe;
        if (li >= 128)
          wide_list[atomicAdd(&s_nw, 1u)] = (uint16_t)r;
        else
          narrow_list[atomicAdd(&s_nn, 1u)] = (uint16_t)r;
      }
      run_p += tp;
      run_e += te;
    }
    if (tid == 0) {
      s_tot[0] = run_p;
      s_tot[1] = run_e;
    }
  }
  __syncthreads();
  if (s_bad || s_tot[0] > F_GCAP || (a.want_enc && s_tot[1] > F_ARENA_W)) {
    defer();  // a term of more than REG_CAP values, or lists that do not fit the slots
    return;
  }

  // ---------------- (5) sources of every term -> its gather slot ----------------
  // (the key windows are dead: the gather slots take their place)
#pragma unroll
  for (int j = 0; j < F_PER; j++) {
    const uint32_t i = tid + j * F_THREADS;
    if (i < W) {
      const uint32_t g = og[j] >> 20;
      const uint32_t* src = reinterpret_cast<const uint32_t*>(smem + ps[j]);
      uint32_t* dst = gather + pbase[g] + (og[j] & 0xFFFFFu);
      const uint32_t n = pl[j];
      uint32_t t = 0;
#pragma unroll 1
      for (; t + 4 <= n; t += 4) {
        const uint32_t x0 = src[t], x1 = src[t + 1], x2 = src[t + 2], x3 = src[t + 3];
        dst[t] = x0;
        dst[t + 1] = x1;
        dst[t + 2] = x2;
        dst[t + 3] = x3;
      }
      if (t < n) {
        const uint32_t x0 = src[t];
        const uint32_t x1 = t + 1 < n ? src[t + 1] : 0u;
        const uint32_t x2 = t + 2 < n ? src[t + 2] : 0u;
        dst[t] = x0;
        if (t + 1 < n) dst[t + 1] = x1;
        if (t + 2 < n) dst[t + 2] = x2;
      }
    }
  }
  __syncthreads();  // areas A and C are dead: they become the `_val` arena

  // ---------------- (6) union + dedup + filter + encode ----------------
  // Work items, longest first: a term of 128 .. 256 values takes a whole warp (eight values per
  // lane), shorter terms go two to a warp (one per 16-lane group).  All items of a bucket
  // usually fit one round of the CTA's warps, so the phase lasts as long as ONE union.
  uint32_t* const arena = reinterpret_cast<uint32_t*>(smem + OFF_A);
  {
    const unsigned half = lane >> 4, hl = lane & 15u;
    const uint32_t nw = s_nw, nn = s_nn;
    const uint32_t items = nw + ((nn + 1) >> 1);
#pragma unroll 1
    for (uint32_t it = warp; it < items; it += F_WARPS) {
      if (it < nw) {
        const uint32_t r = wide_list[it];
        const uint32_t me = order[r];
        const uint32_t c = cg[me];
        uint32_t* const wslot = gather + pbase[me];
        uint32_t* const weslot = arena + ebase[me];
        const uint32_t outn = union_blocked<32>(wslot, wslot, c & 0xFFFFFu, (c >> 20) > 1, a.rem);
        uint32_t enc = 0;
        if (a.want_enc && outn) enc = encode_shared_warp(wslot, outn, weslot);
        if (lane == 0) rres[r] = outn | (enc << 16);
      } else {
        const uint32_t q = 2 * (it - nw) + half;
        const bool has = q < nn;
        const uint32_t r = has ? narrow_list[q] : 0u;
        const uint32_t me = has ? order[r] : 0u;
        const uint32_t c = has ? cg[me] : 0u;
        uint32_t* const slot = gather + (has ? pbase[me] : 0u);
        uint32_t* const eslot = arena + (has ? ebase[me] : 0u);
        const uint32_t outn = union_blocked<16>(slot, slot, c & 0xFFFFFu, (c >> 20) > 1, a.rem);
        uint32_t enc = 0;
        if (a.want_enc) enc = encode_small_blocked<16>(slot, outn, eslot);
        if (has && hl == 0) rres[r] = outn | (enc << 16);
      }
      __syncwarp();
    }
  }
  __syncthreads();

  // ---------------- (7) surviving terms, densely, in merged order ----------------
  // pfx[r] (exclusive, packed): terms | postings << 11 | words << 24 | term bytes << 38
  const bool keep_empty = a.keep_empty != 0;
  auto packed = [&](uint32_t r) -> uint64_t {
    const uint32_t res = rres[r];
    const uint32_t cnt = res & 0xFFFFu, enc = res >> 16;
    if (!(cnt || keep_empty)) return 0ull;
    return 1ull | ((uint64_t)cnt << 11) | ((uint64_t)enc << 24) | ((uint64_t)tlen[order[r]] << 38);
  };
  if (D <= 64) {
    if (warp == 0) {
      const uint64_t v0 = lane < D ? packed(lane) : 0ull;
      const uint64_t v1 = lane + 32 < D ? packed(lane + 32) : 0ull;
      const uint64_t i0 = warp_inclusive_scan(v0);
      const uint64_t t0 = __shfl_sync(0xffffffffu, i0, 31);
      const uint64_t i1 = warp_inclusive_scan(v1) + t0;
      if (lane < D) pfx[lane] = i0 - v0;
      if (lane + 32 < D) pfx[lane + 32] = i1 - v1;
      if (lane == 31) s_total = i1;
    }
  } else {
    uint64_t run = 0;
    for (uint32_t base = 0; base < D; base += F_THREADS) {
      const uint32_t r = base + tid;
      const uint64_t v = r < D ? packed(r) : 0ull;
      uint64_t tot;
      const uint64_t ex = block_exclusive_scan(v, s_ws64, tot);
      if (r < D) pfx[r] = run + ex;
      run += tot;
    }
    if (tid == 0) s_total = run;
  }
  __syncthreads();
  {
    const uint64_t P0 = a.bk_P[b], E0 = a.bk_E[b], T0 = a.bk_TB[b];
    uint8_t* const o_tb = a.st_tb + T0;
    uint32_t* const o_enc = a.st_enc + E0;
    uint32_t* const o_post = a.st_post + P0;
#pragma unroll 1
    for (uint32_t r = warp; r < D; r += F_WARPS) {
      const uint32_t res = rres[r];
      const uint32_t cnt = res & 0xFFFFu, enc = res >> 16;
      if (!(cnt || keep_empty)) continue;
      const uint32_t me = order[r];
      const uint64_t x = pfx[r];
      const uint32_t t = (uint32_t)x & 0x7FFu, po = (uint32_t)(x >> 11) & 0x1FFFu,
                     eo = (uint32_t)(x >> 24) & 0x3FFFu, to = (uint32_t)(x >> 38);
      const uint32_t n = tlen[me];
      if (lane == 0) {
        a.st_toff[rec_base + t] = to;
        if (a.want_enc) a.st_eoff[rec_base + t] = eo;
        if (a.want_dec) a.st_poff[rec_base + t] = po;
      }
      const uint8_t* tsrc = smem + OFF_B + tsm[me];
      for (uint32_t i = lane; i < n; i += 32) o_tb[to + i] = tsrc[i];
      if (a.want_enc) {
        const uint32_t* esrc = arena + ebase[me];
        for (uint32_t i = lane; i < enc; i += 32) o_enc[eo + i] = esrc[i];
      }
      if (a.want_dec) {
        const uint32_t* dsrc = gather + pbase[me];
        for (uint32_t i = lane; i < cnt; i += 32) o_post[po + i] = dsrc[i];
      }
    }
  }
  if (tid == 0) {
    const uint64_t x = s_total;
    a.bk_D[b] = D;
    a.bk_mode[b] = K12F_DENSE;
    a.bk_raw[0ull * a.nb1 + b] = x & 0x7FFu;
    a.bk_raw[1ull * a.nb1 + b] = x >> 38;
    a.bk_raw[2ull * a.nb1 + b] = (x >> 11) & 0x1FFFu;
    a.bk_raw[3ull * a.nb1 + b] = (x >> 24) & 0x3FFFu;
  }
}

bool k12f_supported(int k) {
  // one thread per segment in the header, 4 k copy descriptors in 16 * F_CAP_I bytes
  return k >= 1 && k <= (int)F_MAXK && 4 * k <= (int)F_CAP_I && k <= F_THREADS;
}

int k12f_launch(const K12fArgs& a, uint32_t n_buckets, cudaStream_t s) {
  const size_t smem = k12f_smem_bytes(a.k);
  static size_t attr = 0;
  if (smem > attr) {
    const size_t want = k12f_smem_bytes((int)F_MAXK);
    II2_CUDA_TRY(cudaFuncSetAttribute(k12f_bucket_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)want));
    attr = want;
  }
  II2_LAUNCH_CHAIN(k12f_bucket_kernel, n_buckets, F_THREADS, smem, s, a);
  return II2_OK;
}

}  // namespace ii2
