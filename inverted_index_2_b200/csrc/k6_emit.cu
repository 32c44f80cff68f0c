// k6_emit.cu — emit the merged segment / read result from K12's per-term records.
//
// Replaces the writer half of the merge loop: empty-term drop (shard.go:192-194) and
// Writer.Append (file/writer.go:32-59: FST output = running valuesOffset, `_val` = one intcomp
// stream per term, little-endian words, no framing); for reads, the TermValues the iterator
// would yield.  Everything was computed by K12 — this kernel only places it: one CTA per
// bucket walks the bucket's records in chunks of 256, a block scan over the surviving terms
// gives every term its output slots (bucket bases come from the bucket-level scan), then warps
// copy term bytes, encoded words and/or decoded postings.  Pure HBM copy work.
#include <algorithm>

#include "keys.cuh"
#include "union.cuh"

namespace ii2 {

constexpr int K6_THREADS = 256;
constexpr int K6_WARPS = K6_THREADS / 32;
constexpr uint32_t K6_PENDING = 0xFFFFFFFFu;

struct K6Args {
  const SegDesc* segs;
  int k;
  const uint64_t* bk_pos;
  const uint32_t* bk_D;
  const GroupRec* recs;
  const uint32_t* tmp_enc;
  const uint64_t* bk_out;  // [4][nb1] exclusive prefixes
  uint32_t nb1;
  const uint32_t* list;    // or: one bucket per CTA, the buckets the fused kernel deferred
  int want_dec, want_enc, keep_empty;
  uint8_t* o_term_bytes;
  uint32_t* o_term_off;
  uint32_t* o_post;
  uint64_t* o_post_off;
  uint32_t* o_val_words;
  uint64_t* o_val_off;
};

struct K6Work {
  const uint8_t* tsrc;
  const uint32_t* dsrc;
  const uint32_t* esrc;
  uint64_t post_dst;
  uint64_t enc_dst;
  uint32_t tdst;
  uint32_t tlen;
  uint32_t cnt;
  uint32_t enc;
};

constexpr uint32_t K6_MAX_GROUP = 32;  // buckets per CTA

// One CTA places the records of `group` consecutive buckets: their records, bucket after
// bucket, form one flat sequence (buckets are in merged order and bk_out is the exclusive
// prefix over buckets, so the running output positions simply continue across the buckets of
// the group).  About 256 records per CTA: one set of block scans per 256 terms.
constexpr int K6_MIN_CTAS = 6;
__global__ void __launch_bounds__(K6_THREADS, K6_MIN_CTAS) k6_emit_kernel(const K6Args a, uint32_t group,
                                                             uint32_t n_buckets) {
  pdl_enter();
  __shared__ K6Work s_work[K6_THREADS];
  __shared__ uint64_t s_ws64[K6_WARPS + 2];
  __shared__ uint32_t s_pref[K6_MAX_GROUP + 1];
  __shared__ uint64_t s_base[K6_MAX_GROUP];
  const uint32_t tid = threadIdx.x, b0 = a.list ? a.list[blockIdx.x] : blockIdx.x * group;
  const uint32_t nb = a.list ? 1u : min(group, n_buckets - b0);
  if (tid < 32) {
    const uint32_t d = tid < nb ? a.bk_D[b0 + tid] : 0u;
    const uint32_t inc = warp_inclusive_scan(d);
    if (tid < nb) {
      s_pref[tid + 1] = inc;
      s_base[tid] = a.bk_pos[b0 + tid];
    }
    if (tid == 0) s_pref[0] = 0;
  }
  __syncthreads();
  const uint32_t nrec = s_pref[nb];
  uint64_t run_t = a.bk_out[0ull * a.nb1 + b0];
  uint64_t run_tb = a.bk_out[1ull * a.nb1 + b0];
  uint64_t run_p = a.bk_out[2ull * a.nb1 + b0];
  uint64_t run_e = a.bk_out[3ull * a.nb1 + b0];
  for (uint32_t q = 0; q < nrec; q += K6_THREADS) {
    const uint32_t r = q + tid;
    GroupRec g;
    g.cnt = 0;
    g.enc = 0;
    g.tlen = 0;
    uint32_t surv = 0;
    if (r < nrec) {
      uint32_t j = 0;  // bucket of flat record r
      while (s_pref[j + 1] <= r) j++;
      g = a.recs[s_base[j] + (r - s_pref[j])];
      surv = (g.cnt != K6_PENDING && (g.cnt || a.keep_empty)) ? 1u : 0u;
    }
    const uint32_t tl = surv ? g.tlen : 0u;
    const uint32_t cnt = surv ? g.cnt : 0u;
    const uint32_t enc = surv ? g.enc : 0u;
    // (terms, term bytes) share one scan; postings and words can be large, one each
    uint64_t tot_a, tot_p = 0, tot_e = 0;
    const uint64_t ex_a = block_exclusive_scan<uint64_t>((uint64_t)surv | ((uint64_t)tl << 32),
                                                         s_ws64, tot_a);
    const uint64_t ex_p = a.want_dec ? block_exclusive_scan<uint64_t>(cnt, s_ws64, tot_p) : 0ull;
    const uint64_t ex_e = a.want_enc ? block_exclusive_scan<uint64_t>(enc, s_ws64, tot_e) : 0ull;
    const uint32_t n_surv = (uint32_t)tot_a;
    if (surv) {
      const uint64_t t = run_t + (uint32_t)ex_a;
      K6Work w;
      int s;
      uint32_t idx;
      locate_instance(a.segs, a.k, g.inst, s, idx);
      w.tsrc = a.segs[s].tb + a.segs[s].toff[idx];
      w.tlen = tl;
      w.tdst = (uint32_t)(run_tb + (ex_a >> 32));
      w.cnt = cnt;
      w.enc = enc;
      w.dsrc = reinterpret_cast<const uint32_t*>(g.dec);
      w.esrc = reinterpret_cast<const uint32_t*>(g.eoff);
      w.post_dst = run_p + ex_p;
      w.enc_dst = run_e + ex_e;
      s_work[(uint32_t)ex_a] = w;
      a.o_term_off[t] = w.tdst;
      if (a.want_dec) a.o_post_off[t] = w.post_dst;
      if (a.want_enc) a.o_val_off[t] = 4ull * w.enc_dst;
    }
    __syncthreads();
    // A term is ~15 bytes + ~100 words: with one load per lane in flight the warp pays a full
    // memory round trip per 32 words (source and destination may alias as far as the compiler
    // knows, so it keeps load -> store -> load in order).  The first 128 words of both streams
    // and the first 32 term bytes are requested before anything is stored.
    for (uint32_t h = warp_id(); h < n_surv; h += K6_WARPS) {
      const K6Work w = s_work[h];
      const unsigned lane = lane_id();
      uint8_t tb0 = 0;
      uint32_t ev[4], dv[4];
      if (lane < w.tlen) tb0 = __ldg(w.tsrc + lane);
      if (a.want_enc) {
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (u * 32 + lane < w.enc) ev[u] = __ldg(w.esrc + u * 32 + lane);
      }
      if (a.want_dec) {
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (u * 32 + lane < w.cnt) dv[u] = __ldg(w.dsrc + u * 32 + lane);
      }
      if (lane < w.tlen) a.o_term_bytes[w.tdst + lane] = tb0;
      if (a.want_enc) {
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (u * 32 + lane < w.enc) a.o_val_words[w.enc_dst + u * 32 + lane] = ev[u];
      }
      if (a.want_dec) {
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (u * 32 + lane < w.cnt) a.o_post[w.post_dst + u * 32 + lane] = dv[u];
      }
      // the rest of a long term / a heavy term's streams, four requests at a time
      for (uint32_t i = 32 + lane; i < w.tlen; i += 32) a.o_term_bytes[w.tdst + i] = __ldg(w.tsrc + i);
      if (a.want_enc)
        for (uint32_t base = 128; base < w.enc; base += 128) {
#pragma unroll
          for (int u = 0; u < 4; u++)
            if (base + u * 32 + lane < w.enc) ev[u] = __ldg(w.esrc + base + u * 32 + lane);
#pragma unroll
          for (int u = 0; u < 4; u++)
            if (base + u * 32 + lane < w.enc) a.o_val_words[w.enc_dst + base + u * 32 + lane] = ev[u];
        }
      if (a.want_dec)
        for (uint32_t base = 128; base < w.cnt; base += 128) {
#pragma unroll
          for (int u = 0; u < 4; u++)
            if (base + u * 32 + lane < w.cnt) dv[u] = __ldg(w.dsrc + base + u * 32 + lane);
#pragma unroll
          for (int u = 0; u < 4; u++)
            if (base + u * 32 + lane < w.cnt) a.o_post[w.post_dst + base + u * 32 + lane] = dv[u];
        }
    }
    run_t += n_surv;
    run_tb += tot_a >> 32;
    run_p += tot_p;
    run_e += tot_e;
    __syncthreads();
  }
  // terminal offsets, written once by the CTA of the last bucket
  if (b0 + nb == n_buckets && tid == 0) {
    a.o_term_off[run_t] = (uint32_t)run_tb;
    if (a.want_dec) a.o_post_off[run_t] = run_p;
  }
}

// ---- dense buckets (K12f) ---------------------------------------------------------------------
// The fused kernel left bucket b finished and dense in its staging areas; its place in the
// result is the bucket-level prefix.  One warp per bucket: three contiguous copies (term bytes,
// `_val` words, decoded postings) with 16-byte stores on the destination's alignment, and the
// per-term offsets rebased.  Pure HBM copy work.
struct K6DenseArgs {
  const uint64_t* bk_pos;
  const uint64_t* bk_P;
  const uint64_t* bk_E;
  const uint64_t* bk_TB;
  const uint32_t* bk_mode;
  const uint64_t* bk_raw;  // [4][nb1] per bucket: terms, term bytes, postings, words
  const uint64_t* bk_out;  // exclusive prefixes of bk_raw
  uint32_t nb1;
  int want_dec, want_enc;
  const uint8_t* st_tb;
  const uint32_t* st_toff;
  const uint32_t* st_eoff;
  const uint32_t* st_poff;
  const uint32_t* st_enc;
  const uint32_t* st_post;
  uint8_t* o_term_bytes;
  uint32_t* o_term_off;
  uint32_t* o_post;
  uint64_t* o_post_off;
  uint32_t* o_val_words;
  uint64_t* o_val_off;
};

// n words src -> dst by one warp: scalar head up to the destination's 16-byte boundary, then one
// 128-bit store per lane (four coalesced word loads: the source has its own phase), two in flight
__device__ __forceinline__ void warp_copy_words(uint32_t* __restrict__ dst,
                                                const uint32_t* __restrict__ src, uint32_t n) {
  const unsigned lane = lane_id();
  uint32_t head = (uint32_t)(((16u - (reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u) >> 2);
  head = head < n ? head : n;
  if (lane < head) dst[lane] = __ldg(src + lane);
  const uint32_t nvec = (n - head) >> 2;
  uint4* d4 = reinterpret_cast<uint4*>(dst + head);
  const uint32_t* s4 = src + head;
  uint32_t v = lane;
  for (; v + 32 < nvec; v += 64) {
    const uint32_t e0 = 4 * v, e1 = 4 * (v + 32);
    const uint4 x = make_uint4(__ldg(s4 + e0), __ldg(s4 + e0 + 1), __ldg(s4 + e0 + 2), __ldg(s4 + e0 + 3));
    const uint4 y = make_uint4(__ldg(s4 + e1), __ldg(s4 + e1 + 1), __ldg(s4 + e1 + 2), __ldg(s4 + e1 + 3));
    d4[v] = x;
    d4[v + 32] = y;
  }
  if (v < nvec) {
    const uint32_t e0 = 4 * v;
    d4[v] = make_uint4(__ldg(s4 + e0), __ldg(s4 + e0 + 1), __ldg(s4 + e0 + 2), __ldg(s4 + e0 + 3));
  }
  const uint32_t tail0 = head + 4 * nvec;
  if (tail0 + lane < n) dst[tail0 + lane] = __ldg(src + tail0 + lane);
}

// n bytes: byte head up to the destination's 4-byte boundary, then one 32-bit store per lane
__device__ __forceinline__ void warp_copy_bytes(uint8_t* __restrict__ dst,
                                                const uint8_t* __restrict__ src, uint32_t n) {
  const unsigned lane = lane_id();
  uint32_t head = (uint32_t)((4u - (reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u);
  head = head < n ? head : n;
  if (lane < head) dst[lane] = __ldg(src + lane);
  const uint32_t nw = (n - head) >> 2;
  for (uint32_t w = lane; w < nw; w += 32) {
    const uint8_t* p = src + head + 4 * w;
    const uint32_t x = (uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) |
                       ((uint32_t)__ldg(p + 2) << 16) | ((uint32_t)__ldg(p + 3) << 24);
    *reinterpret_cast<uint32_t*>(dst + head + 4 * w) = x;
  }
  const uint32_t tail0 = head + 4 * nw;
  if (tail0 + lane < n) dst[tail0 + lane] = __ldg(src + tail0 + lane);
}

__global__ void __launch_bounds__(K6_THREADS) k6_dense_kernel(const K6DenseArgs a, uint32_t n_buckets) {
  pdl_enter();
  const uint32_t b = blockIdx.x * K6_WARPS + warp_id();
  if (b >= n_buckets) return;
  const unsigned lane = lane_id();
  const uint64_t T0 = a.bk_out[0ull * a.nb1 + b], TB0 = a.bk_out[1ull * a.nb1 + b],
                 P0 = a.bk_out[2ull * a.nb1 + b], E0 = a.bk_out[3ull * a.nb1 + b];
  if (a.bk_mode[b] == K12F_DENSE) {
    const uint32_t T = (uint32_t)a.bk_raw[0ull * a.nb1 + b], TB = (uint32_t)a.bk_raw[1ull * a.nb1 + b],
                   P = (uint32_t)a.bk_raw[2ull * a.nb1 + b], E = (uint32_t)a.bk_raw[3ull * a.nb1 + b];
    const uint64_t pos = a.bk_pos[b];
    for (uint32_t t = lane; t < T; t += 32) {
      a.o_term_off[T0 + t] = (uint32_t)TB0 + a.st_toff[pos + t];
      if (a.want_enc) a.o_val_off[T0 + t] = 4ull * (E0 + a.st_eoff[pos + t]);
      if (a.want_dec) a.o_post_off[T0 + t] = P0 + a.st_poff[pos + t];
    }
    warp_copy_bytes(a.o_term_bytes + TB0, a.st_tb + a.bk_TB[b], TB);
    if (a.want_enc) warp_copy_words(a.o_val_words + E0, a.st_enc + a.bk_E[b], E);
    if (a.want_dec) warp_copy_words(a.o_post + P0, a.st_post + a.bk_P[b], P);
  }
  // terminal offsets: T0 .. of the one-past-the-end bucket row are the totals
  if (b + 1 == n_buckets && lane == 0) {
    const uint64_t T = a.bk_out[0ull * a.nb1 + n_buckets];
    a.o_term_off[T] = (uint32_t)a.bk_out[1ull * a.nb1 + n_buckets];
    if (a.want_dec) a.o_post_off[T] = a.bk_out[2ull * a.nb1 + n_buckets];
  }
}

static void k6_dense_args(const MergePlan& plan, const UnionOut& u, const EmitOut& out, K6DenseArgs& d) {
  const uint32_t N = plan.n_total;
  d.bk_pos = plan.bk_pos();
  d.bk_P = plan.bk_P();
  d.bk_E = plan.bk_E();
  d.bk_TB = plan.bk_TB();
  d.bk_mode = u.bk_mode.p;
  d.bk_raw = u.bk_raw.p;
  d.bk_out = u.bk_out.p;
  d.nb1 = plan.n_buckets + 1;
  d.want_dec = u.want_dec ? 1 : 0;
  d.want_enc = u.want_enc ? 1 : 0;
  d.st_tb = u.st_tb.p;
  d.st_toff = u.st_off.p;
  d.st_eoff = u.st_off.p + N;
  d.st_poff = u.st_off.p + 2 * (size_t)N;
  d.st_enc = u.tmp_enc.p;
  d.st_post = u.tmp_post.p;
  d.o_term_bytes = out.term_bytes.p;
  d.o_term_off = out.term_off.p;
  d.o_post = out.post.p;
  d.o_post_off = out.post_off.p;
  d.o_val_words = out.val_words.p;
  d.o_val_off = out.val_off.p;
}

int k6_emit_early(const MergePlan& plan, UnionOut& u, uint64_t n_in, uint64_t tb_in, EmitOut& out,
                  cudaStream_t s) {
  const uint64_t N = plan.n_total;
  II2_TRY(out.term_bytes.alloc(tb_in, s, 32));
  II2_TRY(out.term_off.alloc(N + 1, s, 16));
  if (u.want_dec) {
    II2_TRY(out.post.alloc(n_in, s, 16));
    II2_TRY(out.post_off.alloc(N + 1, s, 16));
  }
  if (u.want_enc) {
    II2_TRY(out.val_words.alloc(n_in + n_in / 4 + 6 * N + 16, s, 16));
    II2_TRY(out.val_off.alloc(N, s, 16));
  }
  K6DenseArgs d;
  k6_dense_args(plan, u, out, d);
  ProfScope scope("k6_emit", s);
  II2_LAUNCH_CHAIN(k6_dense_kernel, div_up(plan.n_buckets, K6_WARPS), K6_THREADS, 0, s, d, plan.n_buckets);
  u.emitted_early = true;
  return II2_OK;
}

int k6_emit(const MergePlan& plan, const UnionOut& u, EmitOut& out, cudaStream_t s) {
  const uint64_t T = u.h_totals[0], TB = u.h_totals[1], P = u.h_totals[2], E = u.h_totals[3];
  if (TB >= (1ull << 32)) {
    set_last_error("merged term dictionary exceeds 4 GiB of term bytes");
    return II2_ERR_UNSUPPORTED;
  }
  if (u.emitted_early && u.n_def == 0) {  // every bucket was placed by k6_emit_early: exact sizes only
    out.term_bytes.n = TB;
    out.term_off.n = T + 1;
    if (u.want_dec) {
      out.post.n = P;
      out.post_off.n = T + 1;
    }
    if (u.want_enc) {
      out.val_words.n = E;
      out.val_off.n = T;
    }
    return II2_OK;
  }
  II2_TRY(out.term_bytes.alloc(TB, s, 32));
  II2_TRY(out.term_off.alloc(T + 1, s, 16));
  if (u.want_dec) {
    II2_TRY(out.post.alloc(P, s, 16));
    II2_TRY(out.post_off.alloc(T + 1, s, 16));
  }
  if (u.want_enc) {
    II2_TRY(out.val_words.alloc(E, s, 16));
    II2_TRY(out.val_off.alloc(T, s, 16));
  }
  K6Args a;
  a.segs = plan.segs;
  a.k = plan.k;
  a.bk_pos = plan.bk_pos();
  a.bk_D = u.bk_D.p;
  a.recs = u.recs.p;
  a.tmp_enc = u.tmp_enc.p;
  a.bk_out = u.bk_out.p;
  a.nb1 = plan.n_buckets + 1;
  a.list = nullptr;
  a.want_dec = u.want_dec ? 1 : 0;
  a.want_enc = u.want_enc ? 1 : 0;
  a.keep_empty = u.keep_empty ? 1 : 0;
  a.o_term_bytes = out.term_bytes.p;
  a.o_term_off = out.term_off.p;
  a.o_post = out.post.p;
  a.o_post_off = out.post_off.p;
  a.o_val_words = out.val_words.p;
  a.o_val_off = out.val_off.p;
  ProfScope scope("k6_emit", s);
  if (u.fused) {
    K6DenseArgs d;
    k6_dense_args(plan, u, out, d);
    II2_LAUNCH_CHAIN(k6_dense_kernel, div_up(plan.n_buckets, K6_WARPS), K6_THREADS, 0, s, d, plan.n_buckets);
    if (u.n_def) {  // the buckets the general kernels ran: one CTA each, from their records
      a.list = u.def_list.p;
      II2_LAUNCH_CHAIN(k6_emit_kernel, u.n_def, K6_THREADS, 0, s, a, 1, plan.n_buckets);
    }
    return II2_OK;
  }
  // buckets per CTA: about one CTA-width of records
  const uint64_t tm = u.terms_merged ? u.terms_merged : 1;
  uint32_t group = (uint32_t)std::min<uint64_t>(
      K6_MAX_GROUP, std::max<uint64_t>(1, (uint64_t)K6_THREADS * plan.n_buckets / tm));
  // a small result (a narrow range read) must not end up on a handful of CTAs whose warps walk
  // dozens of terms one after the other: at least ~two CTAs per SM while the buckets last
  group = (uint32_t)std::min<uint64_t>(group, std::max<uint64_t>(1, plan.n_buckets / 296));
  II2_LAUNCH_CHAIN(k6_emit_kernel, div_up(plan.n_buckets, group), K6_THREADS, 0, s, a, group, plan.n_buckets);
  return II2_OK;
}

// min / max term of the merged order (pre-filter, shard.go:176-179) = the smallest first term
// and the largest last term over the segments' windows.  One warp.
__global__ void __launch_bounds__(32)
k6_minmax_kernel(const SegDesc* __restrict__ segs, int k, uint8_t* __restrict__ out) {
  pdl_enter();
  const unsigned lane = lane_id();
  int best[2] = {-1, -1};
  for (int s = lane; s < k; s += 32) {
    const SegDesc sd = segs[s];
    if (sd.hi <= sd.lo) continue;
    if (best[0] < 0 ||
        keyed_compare(keyed_term(sd, sd.lo), keyed_term(segs[best[0]], segs[best[0]].lo)) < 0)
      best[0] = s;
    if (best[1] < 0 ||
        keyed_compare(keyed_term(sd, sd.hi - 1), keyed_term(segs[best[1]], segs[best[1]].hi - 1)) > 0)
      best[1] = s;
  }
  uint32_t at = 8;
  for (int which = 0; which < 2; which++) {
    int b = best[which];
    for (int d = 16; d > 0; d >>= 1) {
      const int o = __shfl_xor_sync(0xffffffffu, b, d);
      if (o >= 0) {
        if (b < 0) {
          b = o;
        } else if (o != b) {
          const uint32_t ib = which ? segs[b].hi - 1 : segs[b].lo, io = which ? segs[o].hi - 1 : segs[o].lo;
          const int c = keyed_compare(keyed_term(segs[o], io), keyed_term(segs[b], ib));
          // ties: the smaller segment index, so every lane converges on the same winner
          if (which ? (c > 0 || (c == 0 && o < b)) : (c < 0 || (c == 0 && o < b))) b = o;
        }
      }
    }
    uint32_t n = 0;
    if (b >= 0) {
      const uint32_t idx = which ? segs[b].hi - 1 : segs[b].lo;
      const uint32_t o = segs[b].toff[idx];
      n = segs[b].toff[idx + 1] - o;
      for (uint32_t i = lane; i < n; i += 32) out[at + i] = segs[b].tb[o + i];
    }
    if (lane == 0) reinterpret_cast<uint32_t*>(out)[which] = n;
    at += n;
  }
}

int k6_minmax(const MergePlan& plan, const UnionOut& u, uint8_t* d_out, cudaStream_t s) {
  (void)u;
  II2_LAUNCH_CHAIN(k6_minmax_kernel, 1, 32, 0, s, plan.segs, plan.k, d_out);
  return II2_OK;
}

}  // namespace ii2
