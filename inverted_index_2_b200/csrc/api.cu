// api.cu — C-ABI entry points for compaction and term-range reads (include/ii2.h):
// resident segments / removed sets / results, the device pipelines, and the host-buffer
// convenience calls that stage through them.
#include <algorithm>
#include <cstdlib>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "codec.cuh"
#include "ingest.cuh"
#include "lookup.cuh"
#include "prefix.cuh"
#include "query.cuh"
#include "handles.cuh"
#include "union.cuh"

using namespace ii2;


namespace {

// ------------------------------------------------------------------ small kernels
__global__ void __launch_bounds__(256)
k_direct_to_lists(const uint64_t* __restrict__ val_off, uint32_t n, uint32_t* __restrict__ post,
                  uint64_t* __restrict__ poff) {
  // direct mode: the FST output is the single posting, truncated to uint32 (file/reader.go:75)
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    post[i] = (uint32_t)val_off[i];
    poff[i] = i;
  }
  if (i == n) poff[n] = n;
}

// max term length, and whether offsets are monotone
__global__ void __launch_bounds__(256)
k_seg_check(const uint32_t* __restrict__ toff, uint32_t n, const uint64_t* __restrict__ poff,
            uint32_t* __restrict__ stats /* [0]=max term len, [1]=bad flag */) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t a = toff[i], b = toff[i + 1];
  if (b < a) atomicExch(&stats[1], 1u);
  else atomicMax(&stats[0], b - a);
  if (poff && poff[i + 1] < poff[i]) atomicExch(&stats[1], 1u);
}

// offsets of a slice of a larger segment: subtract the first one
__global__ void __launch_bounds__(256)
k_rebase_u32(uint32_t* __restrict__ off, uint64_t n, uint32_t first) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) off[i] -= first;
}
__global__ void __launch_bounds__(256)
k_woff32_to_bytes(const uint32_t* __restrict__ w, uint64_t n, uint64_t* __restrict__ b) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) b[i] = 4ull * w[i];
}
__global__ void __launch_bounds__(256)
k_rebase_u64(uint64_t* __restrict__ off, uint64_t n, uint64_t first) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) off[i] -= first;
}

// Slices of many segments staged into shared blocks by one range of the pipelined ii2_merge:
// the k_seg_check tests for all of them in one launch (grid.y = slice).
struct SliceRef {
  const uint32_t* toff;  // [n + 1]
  const uint64_t* poff;  // [n + 1]
  uint32_t n;
  uint32_t pad;
};
__global__ void __launch_bounds__(256)
k_slices_check(const SliceRef* __restrict__ sl, uint32_t* __restrict__ stats) {
  const SliceRef f = sl[blockIdx.y];
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < f.n;
       i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t a = f.toff[i], b = f.toff[i + 1];
    if (b < a) atomicExch(&stats[1], 1u);
    else atomicMax(&stats[0], b - a);
    if (f.poff && f.poff[i + 1] < f.poff[i]) atomicExch(&stats[1], 1u);
  }
}

// `_val` slices of one range of the pipelined ii2_merge (II2_SEG_VAL views): every slice was
// staged at the phase of its source; the decoder wants one array of words with list i at
// [woff[i], woff[i+1]), so the slices are moved back to back (grid.y = slice) ...
struct ValSlice {
  const uint32_t* src;   // staged words of the slice
  const void* off;       // staged FST outputs of its terms: u64 byte offsets or u32 word offsets
  uint64_t first;        // output of the slice's first term, in BYTES
  uint64_t words;        // words of the slice
  uint64_t wbase;        // first word of the slice in the compact array
  uint64_t tbase;        // first list of the slice among the range's `_val` lists
  uint32_t n;            // terms of the slice
  uint32_t off32;        // offsets are u32 word offsets
};
__global__ void __launch_bounds__(256)
k_val_compact(const ValSlice* __restrict__ sl, uint32_t* __restrict__ dst) {
  const ValSlice f = sl[blockIdx.y];
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < f.words;
       i += (uint64_t)gridDim.x * blockDim.x)
    dst[f.wbase + i] = f.src[i];
}
// ... and every term's FST output (file/reader.go:50-52: a run ends where the next one starts,
// the last one at the end of the slice) becomes a word offset into the compact array.
// stats[1] = 1 on an offset that is not 4-byte aligned, not monotone or past the slice.
__global__ void __launch_bounds__(256)
k_val_woff(const ValSlice* __restrict__ sl, uint32_t nslices, uint64_t* __restrict__ woff,
           uint32_t* __restrict__ stats) {
  const ValSlice f = sl[blockIdx.y];
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < f.n;
       i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t b, nb;  // bytes from the start of the segment's `_val`
    if (f.off32) {
      const uint32_t* o = static_cast<const uint32_t*>(f.off);
      b = 4ull * o[i];
      nb = i + 1 < f.n ? 4ull * o[i + 1] : f.first + 4ull * f.words;
    } else {
      const uint64_t* o = static_cast<const uint64_t*>(f.off);
      b = o[i];
      nb = i + 1 < f.n ? o[i + 1] : f.first + 4ull * f.words;
    }
    if ((b & 3u) || b < f.first || nb < b || nb > f.first + 4ull * f.words) {
      atomicExch(&stats[1], 1u);
      b = f.first;
    }
    woff[f.tbase + i] = f.wbase + ((b - f.first) >> 2);
  }
  if (blockIdx.y + 1 == nslices && blockIdx.x == 0 && threadIdx.x == 0)
    woff[f.tbase + f.n] = f.wbase + f.words;  // terminal entry: the slices are back to back
}

// Staging kernel of the pipelined ii2_merge: gathers many host arrays (pinned, mapped into the
// device address space by unified addressing) into device blocks with plain loads over the
// bus.  One launch per term range replaces hundreds of copy-engine requests (measured ~7 us
// of engine time each, more than the small slices take to transfer).
// Reads over the bus are fastest as whole aligned lines (scripts/h2d_micro.cu on B200: 51.5 GB/s
// from a 512-byte aligned source, 46.9 .. 49.6 GB/s at other phases), and a slice starts anywhere
// in its host array.  So a job is laid out over the 512-byte aligned ENVELOPE of its source
// range: vector v of the job is the 16 bytes at (src rounded down to 512) + 16 v, a warp reads
// one aligned 512-byte block, and dst shares the phase of src modulo 512 so the stores are whole
// lines as well.  The vectors that straddle an end of the range (at most two per job) are copied
// byte by byte by their lane, loads first.
struct GatherJob {
  const uint8_t* src;  // host
  uint8_t* dst;        // device, dst = src (mod 512)
  uint64_t bytes;
  uint64_t vec0;       // envelope vectors of the jobs before this one (a multiple of 32)
};
constexpr int kGatherThreads = 256;
constexpr int kGatherUnroll = 4;
constexpr uint64_t kGatherAlign = 512;

// envelope vectors of one job, rounded up to whole warps
static inline uint64_t gather_job_vectors(const void* src, uint64_t bytes) {
  const uint64_t lead = reinterpret_cast<uintptr_t>(src) & (kGatherAlign - 1);
  return (((lead + bytes + 15) >> 4) + 31) & ~31ull;
}

__global__ void __launch_bounds__(kGatherThreads)
k_gather_host(const GatherJob* __restrict__ jobs, uint32_t njobs, uint64_t nvec_total) {
  const uint64_t tile = (uint64_t)kGatherThreads * kGatherUnroll;
  for (uint64_t v0 = (uint64_t)blockIdx.x * tile; v0 < nvec_total; v0 += (uint64_t)gridDim.x * tile) {
    uint4 x[kGatherUnroll];
    uint4* d[kGatherUnroll];
#pragma unroll
    for (int u = 0; u < kGatherUnroll; u++) {
      const uint64_t v = v0 + (uint64_t)u * kGatherThreads + threadIdx.x;
      d[u] = nullptr;
      if (v < nvec_total) {
        uint32_t lo = 0, hi = njobs;  // last job with vec0 <= v (the same job for a whole warp)
        while (hi - lo > 1) {
          const uint32_t mid = (lo + hi) >> 1;
          if (jobs[mid].vec0 <= v)
            lo = mid;
          else
            hi = mid;
        }
        const GatherJob g = jobs[lo];
        const int64_t lead = (int64_t)(reinterpret_cast<uintptr_t>(g.src) & (kGatherAlign - 1));
        const int64_t pos = (int64_t)((v - g.vec0) << 4) - lead;  // of this vector, from src
        if (pos >= 0 && pos + 16 <= (int64_t)g.bytes) {
          x[u] = *reinterpret_cast<const uint4*>(g.src + pos);
          d[u] = reinterpret_cast<uint4*>(g.dst + pos);
        } else if (pos + 16 > 0 && pos < (int64_t)g.bytes) {  // straddles an end of the range
          uint8_t b[16];
#pragma unroll
          for (int i = 0; i < 16; i++) {
            const int64_t q = pos + i;
            b[i] = (q >= 0 && q < (int64_t)g.bytes) ? g.src[q] : (uint8_t)0;
          }
#pragma unroll
          for (int i = 0; i < 16; i++) {
            const int64_t q = pos + i;
            if (q >= 0 && q < (int64_t)g.bytes) g.dst[q] = b[i];
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kGatherUnroll; u++)
      if (d[u]) *d[u] = x[u];
  }
}

__global__ void __launch_bounds__(256)
k_bitmap_set(const uint32_t* __restrict__ sorted, uint64_t n, uint32_t* __restrict__ bitmap,
             uint64_t bitmap_bits) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && sorted[i] < bitmap_bits) atomicOr(&bitmap[sorted[i] >> 5], 1u << (sorted[i] & 31u));
}

// stats[0] = 1 if the list is not ascending (RemovedLists.Values sorts it, removed_list.go:44-54;
// the binary search and the bitmap size both rely on it)
__global__ void __launch_bounds__(256)
k_removed_check(const uint32_t* __restrict__ sorted, uint64_t n, uint32_t* __restrict__ stats) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i + 1 < n;
       i += (uint64_t)gridDim.x * blockDim.x)
    if (sorted[i + 1] < sorted[i]) atomicExch(&stats[0], 1u);
}

// Range windows (K4): lo = first term >= min (vellum Iterator(min) seek, file/reader.go:147),
// hi = first term > max (inclusive right bound, :54-58 and :151-155); then bases.
// A WARP searches 32 ways at a time (warp_partition_point: 4 rounds for 500 k
// terms instead of the 19 dependent probes of a binary search — a small read spent 50 of its
// 270 us there).  The last CTA to finish turns the window widths into instance bases.
// The kernel is the whole host <-> device exchange of the step (a small read is bound by the
// number of launches, not by their work): it reads the segment table and the bounds straight
// from the caller's pinned block, writes the device copy of the table the later kernels use,
// and puts the windows and the postings inside them back into the pinned block.
constexpr uint32_t kBoundsSmem = 4096;
__global__ void __launch_bounds__(256)
k4_windows(const SegDesc* h_segs, SegDesc* d_segs, SegDesc* h_out,
           uint64_t* __restrict__ h_post, int k, const uint8_t* __restrict__ bounds,
           uint32_t minlen, int has_min, uint32_t maxlen, int has_max, uint32_t* ticket) {
  pdl_enter();
  __shared__ uint32_t ws[256 / 32 + 2];
  __shared__ __align__(16) uint8_t s_bounds[kBoundsSmem];
  __shared__ bool s_last;
  // two warps per segment: one finds the start of the window, the other its end, at the same
  // time (each search is a chain of ~8 dependent loads, which is what this kernel's time is)
  __shared__ uint32_t s_hi[4];
  const int s = blockIdx.x * 4 + (warp_id() >> 1);
  const bool upper = warp_id() & 1u;
  SegDesc sd = {};
  if (s < k) sd = h_segs[s];  // (requested before the bounds: two reads over the bus at once)
  const uint8_t* bnd = bounds;
  if (minlen + maxlen <= kBoundsSmem) {  // (longer bounds were uploaded: read them in place)
    for (uint32_t i = threadIdx.x; i < minlen + maxlen; i += 256) s_bounds[i] = bounds[i];
    bnd = s_bounds;
    __syncthreads();
  }
  uint32_t found = 0;
  if (s < k) {
    auto term_vs = [&](uint32_t i, const uint8_t* t, uint32_t nt) {
      const uint32_t o = __ldg(sd.toff + i), n = __ldg(sd.toff + i + 1) - o;
      return term_compare(sd.tb + o, n, t, nt);
    };
    if (!upper)
      found = has_min ? warp_partition_point(0u, sd.n, [&](uint32_t i) {
        return term_vs(i, bnd, minlen) < 0; }) : 0u;
    else
      found = has_max ? warp_partition_point(0u, sd.n, [&](uint32_t i) {
        return term_vs(i, bnd + minlen, maxlen) <= 0; }) : sd.n;
    if (upper && lane_id() == 0) s_hi[warp_id() >> 1] = found;
  }
  __syncthreads();
  if (s < k && !upper && lane_id() == 0) {
    const uint32_t lo = found, hi = max(s_hi[warp_id() >> 1], lo);  // min > max: empty at lo
    sd.lo = lo;
    sd.hi = hi;
    d_segs[s] = sd;  // .base follows below
    h_out[s].lo = lo;
    h_out[s].hi = hi;
    h_post[2 * s] = __ldg(sd.poff + hi) - __ldg(sd.poff + lo);  // sizes the union buffers
    h_post[2 * s + 1] = __ldg(sd.toff + hi) - __ldg(sd.toff + lo);  // and the term bytes
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  uint32_t run = 0;
  for (int base = 0; base < k; base += 256) {
    const int x = base + threadIdx.x;
    const volatile SegDesc* v = d_segs;
    const uint32_t w = x < k ? v[x].hi - v[x].lo : 0u;
    uint32_t tot;
    const uint32_t ex = block_exclusive_scan(w, ws, tot);
    if (x < k) d_segs[x].base = run + ex;
    run += tot;
  }
  if (threadIdx.x == 0) *ticket = 0;  // the next launch finds it zero
}

// ------------------------------------------------------------------ the device pipeline
// segs: resident segments; [min,max] optional; rem optional.
int run_pipeline_impl(ii2_seg* const* segs, int nseg, const uint8_t* min, size_t minlen,
                      bool has_min, const uint8_t* max, size_t maxlen, bool has_max,
                      const ii2_removed* rem, bool want_dec, bool want_enc, bool want_minmax,
                      bool keep_empty, ii2_result** res_out, cudaStream_t s) {
  ProfScope pipe_scope("pipeline_total", s);
  std::unique_ptr<ii2_result> res(new ii2_result());
  res->stream = s;
  res->has_dec = want_dec;
  res->has_enc = want_enc;
  if (nseg < 0 || (nseg > 0 && !segs)) return II2_ERR_INVALID;
  if (nseg > kMaxSegs) {
    set_last_error("%d segments in one call (max %d per pass)", nseg, kMaxSegs);
    return II2_ERR_UNSUPPORTED;
  }
  // segment table, sample bases and range bounds travel through one pinned block so that no
  // pageable copy stalls the stream
  const size_t nsegx = nseg ? nseg : 1;
  const size_t stage_bytes = sizeof(SegDesc) * nsegx + 16 * nsegx + 8 * (nsegx + 1) + minlen + maxlen + 64;
  PinnedBlock stage(stage_bytes);
  if (!stage.p) return II2_ERR_NOMEM;
  SegDesc* h = static_cast<SegDesc*>(stage.p);
  uint64_t* h_post = reinterpret_cast<uint64_t*>(h + nsegx);  // (postings, term bytes) inside every window
  uint32_t* h_sbase = reinterpret_cast<uint32_t*>(h_post + 2 * nsegx);
  uint8_t* h_bounds = reinterpret_cast<uint8_t*>(h_sbase + 2 * (nsegx + 1));
  uint64_t n_total64 = 0, n_in = 0, tb_in = 0;  // instances, postings and term bytes in the windows
  II2_TRY(seg_table(h, segs, nseg, &n_total64));
  if (n_total64 >= (1ull << 32)) {
    set_last_error("more than 2^32-1 term instances in one call");
    return II2_ERR_UNSUPPORTED;
  }
  const RemovedSet rs = removed_set(rem);
  // ---- Read(min == max), decoded output: the whole call is one kernel
  if (nseg > 0 && has_min && has_max && minlen == maxlen && minlen <= kPointMaxTerm &&
      (minlen == 0 || memcmp(min, max, minlen) == 0) && want_dec && !want_enc) {
    if (minlen) memcpy(h_bounds, min, minlen);
    uint64_t* const h_res = pinned_scratch() + 32;
    II2_TRY(k4_point_read(h, nseg, h_bounds, (uint32_t)minlen, rs, keep_empty, res->out, h_res, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    if (h_res[0] == 1) {
      res->T = h_res[1];
      res->TB = res->T ? minlen : 0;
      res->P = h_res[2];
      res->E = 0;
      res->postings_in = h_res[3];
      res->terms_merged = h_res[4] ? 1 : 0;
      res->out.term_bytes.n = res->TB;
      res->out.term_off.n = res->T + 1;
      res->out.post.n = res->P;
      res->out.post_off.n = res->T + 1;
      if (want_minmax && res->terms_merged) {  // pre-filter min / max of the merged order: the term
        res->min_term.assign(reinterpret_cast<const char*>(min), minlen);
        res->max_term = res->min_term;
        res->has_minmax = true;
      }
      *res_out = res.release();
      return II2_OK;
    }
    // more than 4096 values: an ordinary read
  }
  DevBuf<SegDesc> d_segs;
  II2_TRY(d_segs.alloc_scratch(nsegx, s));
  const bool ranged = has_min || has_max;
  if (ranged && nseg) {
    ProfScope win_scope("k4_windows_sync", s);
    DevBuf<uint8_t> d_bounds;
    if (has_min && minlen) memcpy(h_bounds, min, minlen);
    if (has_max && maxlen) memcpy(h_bounds + minlen, max, maxlen);
    const uint8_t* bounds = h_bounds;  // read from the pinned block; long ones are uploaded
    if (minlen + maxlen > kBoundsSmem) {
      II2_TRY(d_bounds.alloc_scratch(minlen + maxlen + 8, s));
      II2_TRY(small_copy(d_bounds.p, h_bounds, minlen + maxlen, s));
      bounds = d_bounds.p;
    }
    uint32_t* const ticket = device_tickets();
    if (!ticket) return II2_ERR_NOMEM;
    II2_LAUNCH_CHAIN(k4_windows, div_up(nseg, 4), 256, 0, s, h, d_segs.p, h, h_post, nseg, bounds,
                     (uint32_t)minlen, has_min ? 1 : 0, (uint32_t)maxlen, has_max ? 1 : 0, ticket);
    // the windows come back: the planner spreads its samples over them
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    n_total64 = 0;
    for (int i = 0; i < nseg; i++) {
      n_total64 += h[i].hi - h[i].lo;
      n_in += h_post[2 * i];
      tb_in += h_post[2 * i + 1];
    }
  } else {  // whole dictionaries
    for (int i = 0; i < nseg; i++) {
      n_in += segs[i]->n_post;
      tb_in += segs[i]->term_bytes_len;
    }
    if (nseg) II2_TRY(small_copy(d_segs.p, h, sizeof(SegDesc) * nseg, s));
  }
  const uint32_t n_total = (uint32_t)n_total64;

  EmitOut& out = res->out;
  if (n_total == 0) {  // nothing in range / no terms at all: empty result
    II2_TRY(out.term_bytes.alloc(0, s, 32));
    II2_TRY(out.term_off.alloc(1, s));
    II2_CUDA_TRY(cudaMemsetAsync(out.term_off.p, 0, 4, s));
    if (want_dec) {
      II2_TRY(out.post.alloc(0, s));
      II2_TRY(out.post_off.alloc(1, s));
      II2_CUDA_TRY(cudaMemsetAsync(out.post_off.p, 0, 8, s));
    }
    if (want_enc) {
      II2_TRY(out.val_words.alloc(0, s));
      II2_TRY(out.val_off.alloc(0, s));
    }
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    *res_out = res.release();
    return II2_OK;
  }

  MergePlan plan;
  plan.k = nseg;
  plan.n_total = n_total;
  plan.segs = d_segs.p;
  II2_TRY(k1_build_plan(plan, h, h_sbase, s));
  UnionOut u;
  // a small read: its result is placed before the host waits for the totals (one round trip
  // less); the arrays are sized by the window's own upper bounds, so only where those are small
  if (ranged && n_total <= 65536 && n_in <= (4u << 20) && tb_in <= (16u << 20)) u.early_out = &out;
  II2_TRY(k12_union(plan, rs, want_dec, want_enc, keep_empty, n_in, tb_in, u, s));
  res->T = u.h_totals[0];
  res->TB = u.h_totals[1];
  res->P = u.h_totals[2];
  res->E = u.h_totals[3];
  res->postings_in = n_in;
  res->terms_merged = u.terms_merged;
  DevBuf<uint8_t> d_mm;
  if (want_minmax) {
    II2_TRY(d_mm.alloc_scratch(8 + 2 * 65536, s));
    II2_TRY(k6_minmax(plan, u, d_mm.p, s));
  }
  II2_TRY(k6_emit(plan, u, out, s));

  if (want_minmax) {
    PinnedBlock mm_blk(8 + 2 * 65536);
    uint8_t* mm = static_cast<uint8_t*>(mm_blk.p);
    if (!mm) return II2_ERR_NOMEM;
    cudaError_t e = small_copy(mm, d_mm.p, 4096, s) == II2_OK ? cudaSuccess : cudaErrorUnknown;
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    uint32_t ln[2] = {0, 0};
    if (e == cudaSuccess) {
      memcpy(ln, mm, 8);
      if (8 + (size_t)ln[0] + ln[1] > 4096) {  // long terms: fetch the rest
        e = cudaMemcpyAsync(mm, d_mm.p, 8 + (size_t)ln[0] + ln[1], cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
      }
    }
    if (e != cudaSuccess) {
      set_last_error("min/max copy: %s", cudaGetErrorString(e));
      return II2_ERR_CUDA;
    }
    res->min_term.assign(reinterpret_cast<const char*>(mm) + 8, ln[0]);
    res->max_term.assign(reinterpret_cast<const char*>(mm) + 8 + ln[0], ln[1]);
    res->has_minmax = u.terms_merged > 0;
  } else {
    II2_CUDA_TRY(cudaStreamSynchronize(s));
  }
  *res_out = res.release();
  return II2_OK;
}

// Runs impl(stream) on the calling thread's stream.  On failure the stream is drained (nothing
// still writes the call's buffers) and *out is zeroed; the call's scratch is released either way.
template <typename Out, typename Impl>
int run_on_stream(Out* out, Impl&& impl) {
  cudaStream_t s = cur_stream();
  const int rc = impl(s);
  if (rc != II2_OK) {
    cudaStreamSynchronize(s);
    memset(out, 0, sizeof(*out));
  }
  arena_reset(s);
  return rc;
}

// Frees the host outputs of a call (ii2_merge_out, ii2_read_out, ii2_prefix_out ...).
template <typename Out>
void host_out_free(Out* o) {
  if (!o) return;
  delete static_cast<HostOwner*>(o->_owner);
  memset(o, 0, sizeof(*o));
}

// Intermediates live in the calling thread's scratch arena for the duration of the call.
int run_pipeline(ii2_seg* const* segs, int nseg, const uint8_t* min, size_t minlen, bool has_min,
                 const uint8_t* max, size_t maxlen, bool has_max, const ii2_removed* rem,
                 bool want_dec, bool want_enc, bool want_minmax, bool keep_empty,
                 ii2_result** res_out) {
  return run_on_stream(res_out, [&](cudaStream_t s) {
    return run_pipeline_impl(segs, nseg, min, minlen, has_min, max, maxlen, has_max, rem, want_dec,
                             want_enc, want_minmax, keep_empty, res_out, s);
  });
}

template <typename T>
int h2d(DevBuf<T>& dst, const T* src, size_t n, cudaStream_t s, size_t pad = 0) {
  II2_TRY(dst.alloc(n, s, pad));
  if (n) II2_CUDA_TRY(cudaMemcpyAsync(dst.p, src, n * sizeof(T), cudaMemcpyHostToDevice, s));
  return II2_OK;
}

template <typename T>
int d2h(T** dst, const T* src, size_t n, HostOwner& own, cudaStream_t s) {
  T* p = own.alloc<T>(n);
  if (!p) return II2_ERR_NOMEM;
  if (n) II2_CUDA_TRY(cudaMemcpyAsync(p, src, n * sizeof(T), cudaMemcpyDeviceToHost, s));
  *dst = p;
  return II2_OK;
}

// reads the accumulated result of k_seg_check (synchronises s)
int seg_check_result(const uint32_t* d_stats, cudaStream_t s) {
  PinnedBlock blk(8);
  uint32_t* hs = static_cast<uint32_t*>(blk.p);
  if (!hs) return II2_ERR_NOMEM;
  hs[0] = hs[1] = 0;
  cudaError_t e = small_copy(hs, d_stats, 8, s) == II2_OK ? cudaSuccess : cudaErrorUnknown;
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  const uint32_t maxlen = hs[0], bad = hs[1];
  if (e != cudaSuccess) {
    set_last_error("segment check: %s", cudaGetErrorString(e));
    return II2_ERR_CUDA;
  }
  if (bad) {
    set_last_error("segment offsets are not monotone");
    return II2_ERR_INVALID;
  }
  if (maxlen > 65535) {
    set_last_error("term of %u bytes (max 65535)", maxlen);
    return II2_ERR_UNSUPPORTED;
  }
  return II2_OK;
}

}  // namespace

// ------------------------------------------------------------------ C-ABI
extern "C" {

// Upload one segment view on stream s.  The offset arrays may belong to a slice of a larger
// segment (term_off[0], post_off[0], val_off[0] != 0): the bytes / values of the slice are
// copied and the offsets rebased on the device.  d_stats != nullptr defers the offset sanity
// check: the check kernel accumulates into d_stats ([0] = max term length, [1] = bad flag) and
// the caller reads it once for many segments (no host synchronisation here for DECODED and
// DIRECT views; `_val` views synchronise to size their decoded lists).
static int seg_upload_impl(const ii2_seg_view* v, cudaStream_t s, uint32_t* d_stats,
                           ii2_seg** seg_out) {
  *seg_out = nullptr;
  const uint64_t n = v->n_terms;
  if (n >= 0xFFFFFFFFull) {
    set_last_error("segment with %llu terms (max 2^32-2)", (unsigned long long)n);
    return II2_ERR_UNSUPPORTED;
  }
  if (n && !v->term_off) return II2_ERR_INVALID;
  const uint32_t tfirst = n ? v->term_off[0] : 0u;
  if (n && v->term_off[n] < tfirst) return II2_ERR_INVALID;
  if (n && v->term_off[n] > tfirst && !v->term_bytes) return II2_ERR_INVALID;
  std::unique_ptr<ii2_seg> g(new ii2_seg());
  g->n_terms = (uint32_t)n;
  g->term_bytes_len = n ? v->term_off[n] - tfirst : 0;
  II2_TRY(h2d(g->tb, v->term_bytes ? v->term_bytes + tfirst : nullptr, (size_t)g->term_bytes_len, s, 32));
  if (n) {
    II2_TRY(h2d(g->toff, v->term_off, (size_t)n + 1, s));
    if (tfirst) {
      k_rebase_u32<<<div_up(n + 1, 256), 256, 0, s>>>(g->toff.p, n + 1, tfirst);
      II2_LAUNCHED();
    }
  } else {
    II2_TRY(g->toff.alloc(1, s));
    II2_CUDA_TRY(cudaMemsetAsync(g->toff.p, 0, 4, s));
  }
  if (v->mode == II2_SEG_DECODED) {
    if (n && !v->post_off) return II2_ERR_INVALID;
    const uint64_t first = n ? v->post_off[0] : 0;
    if (n && v->post_off[n] < first) return II2_ERR_INVALID;
    g->n_post = n ? v->post_off[n] - first : 0;
    if (g->n_post && !v->post) return II2_ERR_INVALID;
    II2_TRY(h2d(g->post, v->post ? v->post + first : nullptr, (size_t)g->n_post, s, 16));
    if (n) {
      II2_TRY(h2d(g->poff, v->post_off, (size_t)n + 1, s));
      if (first) {
        k_rebase_u64<<<div_up(n + 1, 256), 256, 0, s>>>(g->poff.p, n + 1, first);
        II2_LAUNCHED();
      }
    } else {
      II2_TRY(g->poff.alloc(1, s));
      II2_CUDA_TRY(cudaMemsetAsync(g->poff.p, 0, 8, s));
    }
  } else if (v->mode == II2_SEG_DIRECT) {
    if (n && !v->val_off) return II2_ERR_INVALID;
    DevBuf<uint64_t> d_vo;
    II2_TRY(d_vo.alloc_scratch((size_t)n, s));
    if (n)
      II2_CUDA_TRY(cudaMemcpyAsync(d_vo.p, v->val_off, n * 8, cudaMemcpyHostToDevice, s));
    II2_TRY(g->post.alloc(n, s, 16));
    II2_TRY(g->poff.alloc(n + 1, s));
    k_direct_to_lists<<<div_up(n + 1, 256), 256, 0, s>>>(d_vo.p, (uint32_t)n, g->post.p, g->poff.p);
    II2_LAUNCHED();
    g->n_post = n;
  } else if (v->mode == II2_SEG_VAL) {
    if (n && !v->val_off && !v->val_woff32) return II2_ERR_INVALID;
    if (v->val_size && !v->val_bytes) return II2_ERR_INVALID;
    const uint64_t vfirst = !n ? 0 : (v->val_woff32 ? 4ull * v->val_woff32[0] : v->val_off[0]);
    if (vfirst > v->val_size) return II2_ERR_INVALID;
    const uint64_t vsize = v->val_size - vfirst;
    if ((vsize & 3) || (vfirst & 3)) {
      set_last_error("_val size %llu is not a multiple of 4", (unsigned long long)v->val_size);
      return II2_ERR_CORRUPT;
    }
    DevBuf<uint64_t> d_vo, d_woff;
    DevBuf<uint32_t> d_words;
    II2_TRY(d_vo.alloc_scratch((size_t)n, s));
    if (n && v->val_woff32) {  // 32-bit word offsets -> byte offsets
      DevBuf<uint32_t> d_w32;
      II2_TRY(d_w32.alloc_scratch((size_t)n, s));
      II2_CUDA_TRY(cudaMemcpyAsync(d_w32.p, v->val_woff32, n * 4, cudaMemcpyHostToDevice, s));
      k_woff32_to_bytes<<<div_up(n, 256), 256, 0, s>>>(d_w32.p, n, d_vo.p);
      II2_LAUNCHED();
    } else if (n) {
      II2_CUDA_TRY(cudaMemcpyAsync(d_vo.p, v->val_off, n * 8, cudaMemcpyHostToDevice, s));
    }
    if (n && vfirst) {
      k_rebase_u64<<<div_up(n, 256), 256, 0, s>>>(d_vo.p, n, vfirst);
      II2_LAUNCHED();
    }
    II2_TRY(d_words.alloc_scratch(vsize / 4, s, 16));
    if (vsize)
      II2_CUDA_TRY(cudaMemcpyAsync(d_words.p, v->val_bytes + vfirst, vsize, cudaMemcpyHostToDevice, s));
    II2_TRY(val_offsets_to_word_offsets(d_vo.p, n, vsize, d_woff, s));
    uint64_t total = 0;
    II2_TRY(intcomp_decode_dev(d_words.p, d_woff.p, n, g->post, g->poff, &total, s, false));
    g->n_post = total;
  } else {
    set_last_error("unknown segment mode %d", v->mode);
    return II2_ERR_INVALID;
  }
  // sanity: monotone offsets; term lengths must fit the tile kernel's 16-bit length field
  DevBuf<uint32_t> stats;
  uint32_t* st = d_stats;
  if (!st) {
    II2_TRY(stats.alloc_scratch(2, s));
    II2_CUDA_TRY(cudaMemsetAsync(stats.p, 0, 8, s));
    st = stats.p;
  }
  if (n) {
    k_seg_check<<<div_up(n, 256), 256, 0, s>>>(g->toff.p, (uint32_t)n, g->poff.p, st);
    II2_LAUNCHED();
  }
  if (!d_stats) II2_TRY(seg_check_result(st, s));
  *seg_out = g.release();
  return II2_OK;
}

int ii2_seg_upload(const ii2_seg_view* v, ii2_seg** seg_out) {
  if (!v || !seg_out) return II2_ERR_INVALID;
  *seg_out = nullptr;
  II2_TRY(ctx_require());
  cudaStream_t s = cur_stream();
  const int rc = seg_upload_impl(v, s, nullptr, seg_out);
  if (rc != II2_OK) cudaStreamSynchronize(s);
  arena_reset(s);
  return rc;
}

void ii2_seg_release(ii2_seg* seg) {
  if (!seg) return;
  DeviceScope on(seg->device);
  delete seg;
}

int ii2_removed_upload(const uint32_t* removed_sorted, uint64_t nrem, ii2_removed** out) {
  if (!out || (nrem && !removed_sorted)) return II2_ERR_INVALID;
  *out = nullptr;
  II2_TRY(ctx_require());
  cudaStream_t s = cur_stream();
  std::unique_ptr<ii2_removed> r(new ii2_removed());
  if (nrem == 0) removed_sorted = nullptr;
  r->n = nrem;
  II2_TRY(h2d(r->sorted, removed_sorted, (size_t)nrem, s));
  if (nrem) {
    // the caller's list must be ascending (raw C-ABI input: checked, not trusted)
    DevBuf<uint32_t> d_bad;
    II2_TRY(d_bad.alloc_scratch(2, s));
    II2_CUDA_TRY(cudaMemsetAsync(d_bad.p, 0, 8, s));
    k_removed_check<<<(unsigned)std::min<uint64_t>(div_up(nrem, 256), 1184), 256, 0, s>>>(r->sorted.p, nrem, d_bad.p);
    II2_LAUNCHED();
    uint32_t* h_bad = reinterpret_cast<uint32_t*>(pinned_scratch() + 24);
    h_bad[0] = 0;
    II2_TRY(small_copy(h_bad, d_bad.p, 8, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    if (h_bad[0]) {
      arena_reset(s);
      set_last_error("removed list is not sorted ascending");
      return II2_ERR_INVALID;
    }
    // membership bitmap when the id range is small enough to stay L2-friendly (<= 64 MiB)
    const uint64_t maxv = removed_sorted[nrem - 1];
    if (maxv < (1ull << 29) && nrem >= 64) {
      r->bitmap_bits = (maxv + 32) & ~31ull;
      II2_TRY(r->bitmap.alloc(r->bitmap_bits / 32, s));
      II2_CUDA_TRY(cudaMemsetAsync(r->bitmap.p, 0, r->bitmap_bits / 8, s));
      k_bitmap_set<<<div_up(nrem, 256), 256, 0, s>>>(r->sorted.p, nrem, r->bitmap.p, r->bitmap_bits);
      II2_LAUNCHED();
    }
  }
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  *out = r.release();
  return II2_OK;
}

void ii2_removed_release(ii2_removed* rem) {
  if (!rem) return;
  DeviceScope on(rem->device);
  delete rem;
}

int ii2_merge_dev(ii2_seg* const* segs, int nseg, const ii2_removed* rem, uint32_t flags,
                  ii2_result** res) {
  if (!res) return II2_ERR_INVALID;
  *res = nullptr;
  int dev = -1;
  II2_TRY(handles_device(segs, nseg, rem, &dev));
  II2_TRY(ctx_require_device(dev));
  if (flags == 0) flags = II2_RESULT_DECODED;
  // merge: full windows, min/max recorded, emptied terms dropped
  return run_pipeline(segs, nseg, nullptr, 0, false, nullptr, 0, false, rem,
                      (flags & II2_RESULT_DECODED) != 0, (flags & II2_RESULT_ENCODED) != 0, true,
                      false, res);
}

int ii2_read_range_dev(ii2_seg* const* segs, int nseg, const uint8_t* min, size_t minlen,
                       const uint8_t* max, size_t maxlen, const ii2_removed* rem,
                       ii2_result** res) {
  if (!res) return II2_ERR_INVALID;
  *res = nullptr;
  int dev = -1;
  II2_TRY(handles_device(segs, nseg, rem, &dev));
  II2_TRY(ctx_require_device(dev));
  // plain reads keep empty lists (file/writer_test.go:15 round trip); with a removed list the
  // merge-style filter drops emptied terms
  return run_pipeline(segs, nseg, min, minlen, min != nullptr, max, maxlen, max != nullptr, rem,
                      true, false, false, rem == nullptr, res);
}

int ii2_result_info_get(const ii2_result* r, ii2_result_info* info) {
  if (!r || !info) return II2_ERR_INVALID;
  info->terms_count = r->T;
  info->term_bytes = r->TB;
  info->postings_out = r->P;
  info->postings_in = r->postings_in;
  info->terms_merged = r->terms_merged;
  info->val_size = r->E * 4;
  info->d_term_bytes = r->out.term_bytes.p;
  info->d_term_off = r->out.term_off.p;
  info->d_post = r->out.post.p;
  info->d_post_off = r->out.post_off.p;
  info->d_val_bytes = r->out.val_words.p;
  info->d_val_off = r->out.val_off.p;
  return II2_OK;
}

int ii2_result_download_merge(const ii2_result* r, uint32_t flags, ii2_merge_out* o) {
  if (!r || !o) return II2_ERR_INVALID;
  memset(o, 0, sizeof(*o));
  II2_TRY(ctx_require_device(r->device));
  if (!r->has_enc) {
    set_last_error("result was produced without the encoder");
    return II2_ERR_INVALID;
  }
  cudaStream_t s = cur_stream();
  std::unique_ptr<HostOwner> own(new HostOwner());
  II2_TRY(d2h(&o->term_bytes, r->out.term_bytes.p, (size_t)r->TB, *own, s));
  II2_TRY(d2h(&o->term_off, r->out.term_off.p, (size_t)r->T + 1, *own, s));
  II2_TRY(d2h(&o->val_off, r->out.val_off.p, (size_t)r->T, *own, s));
  uint32_t* words = nullptr;
  II2_TRY(d2h(&words, r->out.val_words.p, (size_t)r->E, *own, s));
  o->val_bytes = reinterpret_cast<uint8_t*>(words);
  o->val_size = r->E * 4;
  if ((flags & II2_MERGE_WANT_DECODED) && r->has_dec) {
    II2_TRY(d2h(&o->post, r->out.post.p, (size_t)r->P, *own, s));
    II2_TRY(d2h(&o->post_off, r->out.post_off.p, (size_t)r->T + 1, *own, s));
  }
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  o->terms_count = r->T;
  o->has_minmax = r->has_minmax ? 1 : 0;
  if (r->has_minmax) {
    o->min_term = own->alloc<uint8_t>(r->min_term.size() + 1);
    o->max_term = own->alloc<uint8_t>(r->max_term.size() + 1);
    if (!o->min_term || !o->max_term) return II2_ERR_NOMEM;
    memcpy(o->min_term, r->min_term.data(), r->min_term.size());
    memcpy(o->max_term, r->max_term.data(), r->max_term.size());
    o->min_term_len = (uint32_t)r->min_term.size();
    o->max_term_len = (uint32_t)r->max_term.size();
  }
  o->terms_merged = r->terms_merged;
  o->postings_in = r->postings_in;
  o->postings_out = r->P;
  o->_owner = own.release();
  return II2_OK;
}

int ii2_result_download_read(const ii2_result* r, ii2_read_out* o) {
  if (!r || !o) return II2_ERR_INVALID;
  memset(o, 0, sizeof(*o));
  II2_TRY(ctx_require_device(r->device));
  if (!r->has_dec) return II2_ERR_INVALID;
  cudaStream_t s = cur_stream();
  std::unique_ptr<HostOwner> own(new HostOwner());
  II2_TRY(d2h(&o->term_bytes, r->out.term_bytes.p, (size_t)r->TB, *own, s));
  II2_TRY(d2h(&o->term_off, r->out.term_off.p, (size_t)r->T + 1, *own, s));
  II2_TRY(d2h(&o->post, r->out.post.p, (size_t)r->P, *own, s));
  II2_TRY(d2h(&o->post_off, r->out.post_off.p, (size_t)r->T + 1, *own, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  o->n_terms = r->T;
  o->_owner = own.release();
  return II2_OK;
}

int ii2_result_to_seg(ii2_result* r, ii2_seg** seg_out) {
  if (!r || !seg_out) return II2_ERR_INVALID;
  *seg_out = nullptr;
  if (!r->has_dec || !r->out.post_off.p) return II2_ERR_INVALID;
  if (r->T >= 0xFFFFFFFFull) return II2_ERR_UNSUPPORTED;
  std::unique_ptr<ii2_seg> g(new ii2_seg());
  g->device = r->device;
  g->n_terms = (uint32_t)r->T;
  g->n_post = r->P;
  g->term_bytes_len = r->TB;
  g->tb = std::move(r->out.term_bytes);
  g->toff = std::move(r->out.term_off);
  g->post = std::move(r->out.post);
  g->poff = std::move(r->out.post_off);
  r->has_dec = false;
  r->T = r->TB = r->P = 0;
  *seg_out = g.release();
  return II2_OK;
}

void ii2_result_release(ii2_result* r) {
  if (!r) return;
  DeviceScope on(r->device);
  delete r;
}

int ii2_result_device(const ii2_result* r, int* device) {
  if (!ctx_ready()) {
    set_last_error("ii2_init has not succeeded: no CUDA device bound (there is no CPU fallback)");
    return II2_ERR_NO_DEVICE;
  }
  if (!r || !device) return II2_ERR_INVALID;
  *device = r->device;
  return II2_OK;
}

// ------------------------------------------------------------------ PrefixSearch
static int prefix_search_impl(ii2_seg* const* segs, int nseg, const uint8_t* prefix_bytes,
                              const uint32_t* prefix_off, uint32_t nprefix, ii2_prefix_out* o,
                              cudaStream_t s) {
  ProfScope pipe_scope("prefix_total", s);
  if (nseg > kMaxSegs) {
    set_last_error("%d segments in one call (max %d per pass)", nseg, kMaxSegs);
    return II2_ERR_UNSUPPORTED;
  }
  const size_t pbytes = nprefix ? prefix_off[nprefix] : 0;
  for (uint32_t i = 0; i < nprefix; i++)
    if (prefix_off[i + 1] < prefix_off[i]) return II2_ERR_INVALID;
  // segment table + prefixes through one pinned block (no pageable copy on the stream)
  const size_t nsegx = nseg ? nseg : 1;
  const size_t off_bytes = ((size_t)nprefix + 1) * 4;
  const size_t stage_bytes = sizeof(SegDesc) * nsegx + off_bytes + pbytes + 64;
  PinnedBlock stage(stage_bytes);
  if (!stage.p) return II2_ERR_NOMEM;
  SegDesc* h = static_cast<SegDesc*>(stage.p);
  uint32_t* h_off = reinterpret_cast<uint32_t*>(h + nsegx);
  uint8_t* h_pb = reinterpret_cast<uint8_t*>(h_off + nprefix + 1);
  II2_TRY(seg_table(h, segs, nseg));
  if (nprefix) {
    memcpy(h_off, prefix_off, off_bytes);
    if (pbytes) memcpy(h_pb, prefix_bytes, pbytes);
  } else {
    h_off[0] = 0;
  }
  DevBuf<uint8_t> d_stage;
  II2_TRY(d_stage.alloc_scratch(stage_bytes, s, 32));
  II2_CUDA_TRY(cudaMemcpyAsync(d_stage.p, stage.p, stage_bytes, cudaMemcpyHostToDevice, s));
  const SegDesc* d_segs = reinterpret_cast<const SegDesc*>(d_stage.p);
  const uint32_t* d_off = reinterpret_cast<const uint32_t*>(d_segs + nsegx);
  const uint8_t* d_pb = reinterpret_cast<const uint8_t*>(d_off + nprefix + 1);
  PrefixOut po;
  II2_TRY(k5_prefix_search(d_segs, nseg, d_pb, d_off, nprefix, po, s));
  std::unique_ptr<HostOwner> own(new HostOwner());
  uint32_t* h_matched = nullptr;
  II2_TRY(d2h(&o->values, po.values.p, (size_t)po.total, *own, s));
  II2_TRY(d2h(&o->value_off, po.value_off.p, (size_t)nprefix + 1, *own, s));
  II2_TRY(d2h(&h_matched, po.matched.p, (size_t)(nprefix ? nprefix : 1), *own, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  o->matched = own->alloc<uint8_t>((size_t)nprefix + 1);
  if (!o->matched) return II2_ERR_NOMEM;
  for (uint32_t i = 0; i < nprefix; i++) o->matched[i] = h_matched[i] ? 1 : 0;
  o->n_prefixes = nprefix;
  o->_owner = own.release();
  return II2_OK;
}

int ii2_prefix_search_dev(ii2_seg* const* segs, int nseg, const uint8_t* prefix_bytes,
                          const uint32_t* prefix_off, uint32_t nprefix, ii2_prefix_out* out) {
  if (!out || nseg < 0 || (nseg && !segs) || (nprefix && !prefix_off)) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  int dev = -1;
  II2_TRY(handles_device(segs, nseg, nullptr, &dev));
  II2_TRY(ctx_require_device(dev));
  return run_on_stream(out, [&](cudaStream_t s) {
    return prefix_search_impl(segs, nseg, prefix_bytes, prefix_off, nprefix, out, s);
  });
}

void ii2_prefix_out_free(ii2_prefix_out* o) { host_out_free(o); }

// ------------------------------------------------------------------ batched term lookup
constexpr uint32_t kLookupMaxKey = 65535;  // bytes of one key

static int lookup_impl(ii2_seg* const* segs, int nseg, const uint8_t* key_bytes,
                       const uint32_t* key_off, uint32_t nkeys, const ii2_removed* rem,
                       ii2_lookup_out* o, cudaStream_t s) {
  ProfScope pipe_scope("lookup_total", s);
  if (nseg > kMaxSegs) {
    set_last_error("%d segments in one call (max %d per pass)", nseg, kMaxSegs);
    return II2_ERR_UNSUPPORTED;
  }
  for (uint32_t i = 0; i < nkeys; i++) {
    if (key_off[i + 1] < key_off[i]) return II2_ERR_INVALID;
    if (key_off[i + 1] - key_off[i] > kLookupMaxKey) {
      set_last_error("lookup: key %u is %u bytes long (max %u)", i, key_off[i + 1] - key_off[i],
                     kLookupMaxKey);
      return II2_ERR_UNSUPPORTED;
    }
  }
  const size_t kbytes = nkeys ? key_off[nkeys] : 0;
  if (kbytes && !key_bytes) return II2_ERR_INVALID;
  uint64_t n_post = 0;
  for (int i = 0; i < nseg; i++) {
    if (!segs[i]) return II2_ERR_INVALID;
    n_post += segs[i]->n_post;
  }
  std::unique_ptr<HostOwner> own(new HostOwner());
  o->n_keys = nkeys;
  if (nkeys == 0 || nseg == 0) {  // nothing to find
    o->found = own->alloc<uint8_t>(nkeys);
    o->post_off = own->alloc<uint64_t>((size_t)nkeys + 1);
    o->post = own->alloc<uint32_t>(0);
    if (!o->found || !o->post_off || !o->post) return II2_ERR_NOMEM;
    memset(o->found, 0, nkeys);
    memset(o->post_off, 0, ((size_t)nkeys + 1) * 8);
    o->postings_in = 0;
    o->_owner = own.release();
    return II2_OK;
  }
  // segment table + key offsets + key bytes through one pinned block and one copy
  const size_t off_bytes = ((size_t)nkeys + 1) * 4;
  const size_t stage_bytes = sizeof(SegDesc) * nseg + off_bytes + kbytes + 64;
  PinnedBlock stage(stage_bytes);
  if (!stage.p) return II2_ERR_NOMEM;
  SegDesc* h = static_cast<SegDesc*>(stage.p);
  uint32_t* h_off = reinterpret_cast<uint32_t*>(h + nseg);
  uint8_t* h_kb = reinterpret_cast<uint8_t*>(h_off + nkeys + 1);
  II2_TRY(seg_table(h, segs, nseg));
  memcpy(h_off, key_off, off_bytes);
  if (kbytes) memcpy(h_kb, key_bytes, kbytes);
  DevBuf<uint8_t> d_stage;
  II2_TRY(d_stage.alloc_scratch(stage_bytes, s, 32));
  II2_CUDA_TRY(cudaMemcpyAsync(d_stage.p, stage.p, stage_bytes, cudaMemcpyHostToDevice, s));
  const SegDesc* d_segs = reinterpret_cast<const SegDesc*>(d_stage.p);
  const uint32_t* d_off = reinterpret_cast<const uint32_t*>(d_segs + nseg);
  const uint8_t* d_kb = reinterpret_cast<const uint8_t*>(d_off + nkeys + 1);
  LookupOut lo;
  // plain reads keep empty lists; with a removed set an emptied key is not found (as
  // ii2_read_range_dev)
  II2_TRY(k8_lookup(d_segs, nseg, n_post, d_kb, d_off, nkeys, removed_set(rem), rem == nullptr, lo, s));
  II2_TRY(d2h(&o->found, lo.found.p, nkeys, *own, s));
  II2_TRY(d2h(&o->post_off, lo.post_off.p, (size_t)nkeys + 1, *own, s));
  II2_TRY(d2h(&o->post, lo.post.p, (size_t)lo.total, *own, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  o->postings_in = lo.postings_in;
  o->_owner = own.release();
  return II2_OK;
}

int ii2_lookup_dev(ii2_seg* const* segs, int nseg, const uint8_t* key_bytes,
                   const uint32_t* key_off, uint32_t nkeys, const ii2_removed* rem,
                   ii2_lookup_out* out) {
  if (!out || nseg < 0 || (nseg && !segs) || (nkeys && !key_off)) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  int dev = -1;
  II2_TRY(handles_device(segs, nseg, rem, &dev));
  II2_TRY(ctx_require_device(dev));
  return run_on_stream(out, [&](cudaStream_t s) {
    return lookup_impl(segs, nseg, key_bytes, key_off, nkeys, rem, out, s);
  });
}

void ii2_lookup_out_free(ii2_lookup_out* o) { host_out_free(o); }

// ------------------------------------------------------------------ boolean term queries
constexpr uint32_t kQueryMaxAtom = 65535;      // bytes of one atom (K5's term compare)
constexpr uint32_t kQueryMaxClauseAtoms = 1024;  // sources of one clause union (k2_large_gather)

// off[0 .. n]: starts at 0, monotone, and (last != ~0u) ends at `last`
static bool query_csr_ok(const uint32_t* off, uint32_t n, uint32_t last) {
  if (off[0] != 0) return false;
  for (uint32_t i = 0; i < n; i++)
    if (off[i + 1] < off[i]) return false;
  return last == ~0u || off[n] == last;
}

// The batch's structure, on the host before anything is launched.
static int query_validate(ii2_seg* const* segs, int nseg, const ii2_query_batch* qb) {
  const uint32_t na = qb->natoms, nc = qb->nclauses, nq = qb->nqueries;
  if (!qb->atom_off || !qb->clause_atom_off || !qb->query_clause_off ||
      (na && !qb->atom_kind) || (nc && !qb->clause_excluded)) {
    set_last_error("query: NULL batch array");
    return II2_ERR_INVALID;
  }
  if (!query_csr_ok(qb->atom_off, na, ~0u) || !query_csr_ok(qb->clause_atom_off, nc, na) ||
      !query_csr_ok(qb->query_clause_off, nq, nc)) {
    set_last_error("query: offsets must start at 0, be monotone and end at the next level's count");
    return II2_ERR_INVALID;
  }
  if (qb->atom_off[na] && !qb->atom_bytes) return II2_ERR_INVALID;
  for (uint32_t a = 0; a < na; a++)
    if (qb->atom_kind[a] > II2_ATOM_PREFIX) {
      set_last_error("query: atom %u has unknown kind %u", a, qb->atom_kind[a]);
      return II2_ERR_INVALID;
    }
  for (uint32_t c = 0; c < nc; c++)
    if (qb->clause_excluded[c] > 1) {
      set_last_error("query: clause %u has unknown flag %u", c, qb->clause_excluded[c]);
      return II2_ERR_INVALID;
    }
  for (uint32_t q = 0; q < nq; q++) {
    bool required = false;
    for (uint32_t c = qb->query_clause_off[q]; c < qb->query_clause_off[q + 1] && !required; c++)
      required = qb->clause_excluded[c] == 0;
    if (!required) {
      set_last_error("query %u has no required clause", q);
      return II2_ERR_INVALID;
    }
  }
  for (int i = 0; i < nseg; i++)
    if (!segs[i]) return II2_ERR_INVALID;
  if (nseg > kMaxSegs) {
    set_last_error("%d segments in one call (max %d per pass)", nseg, kMaxSegs);
    return II2_ERR_UNSUPPORTED;
  }
  for (uint32_t a = 0; a < na; a++)
    if (qb->atom_off[a + 1] - qb->atom_off[a] > kQueryMaxAtom) {
      set_last_error("query: atom %u is %u bytes long (max %u)", a,
                     qb->atom_off[a + 1] - qb->atom_off[a], kQueryMaxAtom);
      return II2_ERR_UNSUPPORTED;
    }
  for (uint32_t c = 0; c < nc; c++)
    if (qb->clause_atom_off[c + 1] - qb->clause_atom_off[c] > kQueryMaxClauseAtoms) {
      set_last_error("query: clause %u has %u atoms (max %u)", c,
                     qb->clause_atom_off[c + 1] - qb->clause_atom_off[c], kQueryMaxClauseAtoms);
      return II2_ERR_UNSUPPORTED;
    }
  if ((uint64_t)na * (uint64_t)nseg >= (1ull << 32) || na >= kClauseGroup) {
    set_last_error("query: %u atoms x %d segments exceed 2^32 pairs", na, nseg);
    return II2_ERR_UNSUPPORTED;
  }
  return II2_OK;
}

static int query_impl(ii2_seg* const* segs, int nseg, const ii2_query_batch* qb,
                      const ii2_removed* rem, ii2_query_out* o, cudaStream_t s) {
  ProfScope pipe_scope("query_total", s);
  II2_TRY(query_validate(segs, nseg, qb));
  const uint32_t na = qb->natoms, nc = qb->nclauses, nq = qb->nqueries;
  std::unique_ptr<HostOwner> own(new HostOwner());
  o->n_queries = nq;
  if (nq == 0 || nseg == 0 || na == 0) {  // every clause is empty, so is every result
    o->value_off = own->alloc<uint64_t>((size_t)nq + 1);
    o->values = own->alloc<uint32_t>(0);
    if (!o->value_off || !o->values) return II2_ERR_NOMEM;
    memset(o->value_off, 0, ((size_t)nq + 1) * 8);
    o->clause_values = 0;
    o->_owner = own.release();
    return II2_OK;
  }
  // distinct atoms (kind + bytes), in order of first appearance
  std::vector<uint32_t> uid(na);
  std::vector<uint32_t> u_first;  // an atom of every distinct atom
  size_t ubytes = 0;
  {
    std::unordered_map<std::string, uint32_t> seen;
    seen.reserve(na);
    std::string key;
    for (uint32_t a = 0; a < na; a++) {
      const uint32_t o0 = qb->atom_off[a], n = qb->atom_off[a + 1] - o0;
      key.assign(1, (char)qb->atom_kind[a]);
      if (n) key.append(reinterpret_cast<const char*>(qb->atom_bytes + o0), n);
      auto it = seen.emplace(key, (uint32_t)u_first.size());
      if (it.second) {
        u_first.push_back(a);
        ubytes += n;
      }
      uid[a] = it.first->second;
    }
  }
  const uint32_t nu = (uint32_t)u_first.size();
  uint32_t ng = 0, nsrc = 0;
  for (uint32_t c = 0; c < nc; c++) {
    const uint32_t n = qb->clause_atom_off[c + 1] - qb->clause_atom_off[c];
    if (n >= 2) {
      ng++;
      nsrc += n;
    }
  }
  // segment table, distinct atoms, clauses, query offsets and clause-union sources through one
  // pinned block and one copy; the atoms' list offsets come back into its tail
  size_t cur = 0;
  auto place = [&](size_t bytes) {
    const size_t at = cur;
    cur = (cur + bytes + 15) & ~(size_t)15;
    return at;
  };
  const size_t o_segs = place(sizeof(SegDesc) * nseg);
  const size_t o_gin = place(sizeof(GroupIn) * ng);
  const size_t o_cl = place(sizeof(QueryClause) * nc);
  const size_t o_aoff = place(4 * ((size_t)nu + 1));
  const size_t o_qoff = place(4 * ((size_t)nq + 1));
  const size_t o_grec = place(4 * (size_t)ng);
  const size_t o_gatom = place(4 * (size_t)nsrc);
  const size_t o_kind = place(nu);
  const size_t o_bytes = place(ubytes);
  const size_t stage_bytes = cur;
  const size_t o_voff = place(8 * ((size_t)nu + 1));
  PinnedBlock stage(cur);
  if (!stage.p) return II2_ERR_NOMEM;
  uint8_t* hb = static_cast<uint8_t*>(stage.p);
  II2_TRY(seg_table(reinterpret_cast<SegDesc*>(hb + o_segs), segs, nseg));
  uint32_t* h_aoff = reinterpret_cast<uint32_t*>(hb + o_aoff);
  uint8_t* h_kind = hb + o_kind;
  uint8_t* h_bytes = hb + o_bytes;
  h_aoff[0] = 0;
  for (uint32_t u = 0; u < nu; u++) {
    const uint32_t a = u_first[u], o0 = qb->atom_off[a], n = qb->atom_off[a + 1] - o0;
    if (n) memcpy(h_bytes + h_aoff[u], qb->atom_bytes + o0, n);
    h_aoff[u + 1] = h_aoff[u] + n;
    h_kind[u] = qb->atom_kind[a];
  }
  memcpy(hb + o_qoff, qb->query_clause_off, 4 * ((size_t)nq + 1));
  GroupIn* h_gin = reinterpret_cast<GroupIn*>(hb + o_gin);
  QueryClause* h_cl = reinterpret_cast<QueryClause*>(hb + o_cl);
  uint32_t* h_grec = reinterpret_cast<uint32_t*>(hb + o_grec);
  uint32_t* h_gatom = reinterpret_cast<uint32_t*>(hb + o_gatom);
  for (uint32_t c = 0, g = 0, j = 0; c < nc; c++) {
    const uint32_t a0 = qb->clause_atom_off[c], n = qb->clause_atom_off[c + 1] - a0;
    h_cl[c].excluded = qb->clause_excluded[c];
    if (n == 0) {
      h_cl[c].src = kClauseEmpty;
    } else if (n == 1) {
      h_cl[c].src = uid[a0];
    } else {
      GroupIn gi;
      memset(&gi, 0, sizeof(gi));
      gi.src = j;
      gi.c = n;
      gi.L = 0xFFFFFFFFu;
      h_gin[g] = gi;
      h_grec[g] = g;
      for (uint32_t i = 0; i < n; i++) h_gatom[j++] = uid[a0 + i];
      h_cl[c].src = kClauseGroup | g++;
    }
  }
  DevBuf<uint8_t> d_stage;
  II2_TRY(d_stage.alloc_scratch(stage_bytes, s, 32));
  II2_CUDA_TRY(cudaMemcpyAsync(d_stage.p, stage.p, stage_bytes, cudaMemcpyHostToDevice, s));
  uint8_t* db = d_stage.p;
  QueryDev d;
  d.segs = reinterpret_cast<const SegDesc*>(db + o_segs);
  d.k = nseg;
  d.abytes = db + o_bytes;
  d.aoff = reinterpret_cast<const uint32_t*>(db + o_aoff);
  d.akind = db + o_kind;
  d.nu = nu;
  d.clauses = reinterpret_cast<const QueryClause*>(db + o_cl);
  d.nclauses = nc;
  d.qoff = reinterpret_cast<const uint32_t*>(db + o_qoff);
  d.nq = nq;
  d.gin = reinterpret_cast<const GroupIn*>(db + o_gin);
  d.grec = reinterpret_cast<const uint32_t*>(db + o_grec);
  d.gatom = reinterpret_cast<const uint32_t*>(db + o_gatom);
  d.ngroups = ng;
  d.nsrc = nsrc;
  QueryHost hq;
  hq.clauses = h_cl;
  hq.qoff = qb->query_clause_off;
  hq.gin = h_gin;
  hq.gatom = h_gatom;
  hq.value_off = reinterpret_cast<uint64_t*>(hb + o_voff);
  QueryOut qo;
  II2_TRY(k9_query(d, hq, removed_set(rem), qo, s));
  II2_TRY(d2h(&o->values, qo.values.p, (size_t)qo.total, *own, s));
  II2_TRY(d2h(&o->value_off, qo.value_off.p, (size_t)nq + 1, *own, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  o->clause_values = qo.clause_values;
  o->_owner = own.release();
  return II2_OK;
}

int ii2_query_dev(ii2_seg* const* segs, int nseg, const ii2_query_batch* q, const ii2_removed* rem,
                  ii2_query_out* out) {
  if (!out) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  if (!q || nseg < 0 || (nseg && !segs)) return II2_ERR_INVALID;
  int dev = -1;
  II2_TRY(handles_device(segs, nseg, rem, &dev));
  II2_TRY(ctx_require_device(dev));
  return run_on_stream(out, [&](cudaStream_t s) { return query_impl(segs, nseg, q, rem, out, s); });
}

void ii2_query_out_free(ii2_query_out* o) { host_out_free(o); }

// ------------------------------------------------------------------ ingest batching
static int ingest_impl(const ii2_doc_view* docs, int ndocs, const uint32_t* removed_sorted,
                       uint64_t nrem, uint32_t flags, ii2_merge_out* out, cudaStream_t s) {
  if (ndocs > kMaxSegs) {
    set_last_error("%d documents in one call (max %d per pass)", ndocs, kMaxSegs);
    return II2_ERR_UNSUPPORTED;
  }
  uint64_t N = 0, TB = 0;
  for (int d = 0; d < ndocs; d++) {
    const ii2_doc_view& v = docs[d];
    if (v.n_terms && (!v.term_off || !v.term_bytes)) return II2_ERR_INVALID;
    N += v.n_terms;
    if (v.n_terms) {
      if (v.term_off[v.n_terms] < v.term_off[0]) return II2_ERR_INVALID;
      TB += v.term_off[v.n_terms] - v.term_off[0];
    }
  }
  if (N >= (1ull << 32) || TB >= (1ull << 32)) {
    set_last_error("ingest batch of %llu terms / %llu term bytes (max 2^32-1)",
                   (unsigned long long)N, (unsigned long long)TB);
    return II2_ERR_UNSUPPORTED;
  }
  // offsets rebased to one concatenated buffer, document starts and values: one pinned block
  const size_t off_bytes = ((size_t)N + 1) * 4, doff_bytes = ((size_t)ndocs + 1) * 8;
  const size_t stage_bytes = off_bytes + 8 + doff_bytes + (size_t)ndocs * 4 + 64;
  PinnedBlock stage(stage_bytes);
  if (!stage.p) return II2_ERR_NOMEM;
  uint64_t* h_doff = static_cast<uint64_t*>(stage.p);
  uint32_t* h_vals = reinterpret_cast<uint32_t*>(h_doff + ndocs + 1);
  uint32_t* h_off = h_vals + ndocs + (ndocs & 1);
  DevBuf<uint8_t> d_tb;
  II2_TRY(d_tb.alloc_scratch((size_t)TB, s, 32));
  uint64_t n = 0, b = 0;
  for (int d = 0; d < ndocs; d++) {
    const ii2_doc_view& v = docs[d];
    h_doff[d] = n;
    h_vals[d] = v.value;
    if (!v.n_terms) continue;
    const uint32_t first = v.term_off[0];
    uint32_t max_len = 0;
    for (uint64_t i = 0; i < v.n_terms; i++) {
      if (v.term_off[i + 1] < v.term_off[i]) return II2_ERR_INVALID;
      max_len = std::max(max_len, v.term_off[i + 1] - v.term_off[i]);
      h_off[n + i] = (uint32_t)(b + (v.term_off[i] - first));
    }
    if (max_len > 65535) {
      set_last_error("term of %u bytes (max 65535)", max_len);
      return II2_ERR_UNSUPPORTED;
    }
    const uint64_t nb = v.term_off[v.n_terms] - first;
    if (nb)
      II2_CUDA_TRY(cudaMemcpyAsync(d_tb.p + b, v.term_bytes + first, nb, cudaMemcpyHostToDevice, s));
    n += v.n_terms;
    b += nb;
  }
  h_doff[ndocs] = n;
  h_off[N] = (uint32_t)TB;
  II2_CUDA_TRY(cudaMemsetAsync(d_tb.p + TB, 0, 32, s));
  DevBuf<uint8_t> d_stage;
  II2_TRY(d_stage.alloc_scratch(stage_bytes, s, 32));
  II2_CUDA_TRY(cudaMemcpyAsync(d_stage.p, stage.p, stage_bytes, cudaMemcpyHostToDevice, s));
  const uint64_t* d_doff = reinterpret_cast<const uint64_t*>(d_stage.p);
  const uint32_t* d_vals = reinterpret_cast<const uint32_t*>(d_doff + ndocs + 1);
  const uint32_t* d_off = d_vals + ndocs + (ndocs & 1);
  IngestOut io;
  II2_TRY(k7_ingest_sort(d_tb.p, d_off, d_doff, h_doff, d_vals, ndocs, N, TB, io, s));
  // the documents as resident direct-mode segments: views into the shared buffers
  std::vector<std::unique_ptr<ii2_seg>> owned;
  std::vector<ii2_seg*> list;
  auto view = [](auto& buf, auto* p, size_t cnt) {
    buf.p = p;
    buf.n = cnt;
    buf.scratch = true;  // not owned: never freed through this handle
  };
  for (int d = 0; d < ndocs; d++) {
    const uint64_t f = io.first[d], nt = io.first[d + 1] - f;
    std::unique_ptr<ii2_seg> g(new ii2_seg());
    g->n_terms = (uint32_t)nt;
    g->n_post = nt;
    g->term_bytes_len = io.n_bytes;
    view(g->tb, io.tb.p, (size_t)io.n_bytes);
    view(g->toff, io.toff.p + f, (size_t)nt + 1);
    view(g->post, io.post.p, (size_t)io.n_terms);
    view(g->poff, io.poff.p + f, (size_t)nt + 1);
    list.push_back(g.get());
    owned.push_back(std::move(g));
  }
  ii2_removed* rem = nullptr;
  if (nrem) II2_TRY(ii2_removed_upload(removed_sorted, nrem, &rem));
  std::unique_ptr<ii2_removed> rem_guard(rem);
  ii2_result* res = nullptr;
  II2_TRY(run_pipeline_impl(list.data(), ndocs, nullptr, 0, false, nullptr, 0, false, rem,
                            (flags & II2_MERGE_WANT_DECODED) != 0, true, true, false, &res, s));
  std::unique_ptr<ii2_result> res_guard(res);
  return ii2_result_download_merge(res, flags, out);
}

int ii2_ingest(const ii2_doc_view* docs, int ndocs, const uint32_t* removed_sorted, uint64_t nrem,
               uint32_t flags, ii2_merge_out* out) {
  if (!out || ndocs < 0 || (ndocs && !docs) || (nrem && !removed_sorted)) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  II2_TRY(ctx_require());
  return run_on_stream(out, [&](cudaStream_t s) {
    return ingest_impl(docs, ndocs, removed_sorted, nrem, flags, out, s);
  });
}

void ii2_merge_out_free(ii2_merge_out* o) { host_out_free(o); }

void ii2_read_out_free(ii2_read_out* o) { host_out_free(o); }

// ---- host-buffer entry points: upload, run, download --------------------------------
struct SegList {
  std::vector<ii2_seg*> v;
  // pipelined ii2_merge: the slices of one range live in four shared blocks
  DevBuf<uint8_t> blk_tb;
  DevBuf<uint32_t> blk_toff, blk_post;
  DevBuf<uint64_t> blk_poff;
  DevBuf<SliceRef> blk_ref;
  DevBuf<GatherJob> blk_job;
  // II2_SEG_VAL views: staged `_val` slices and FST outputs, the compact words + word offsets,
  // and the decoded lists of all `_val` segments of the range (shared by their views)
  DevBuf<uint32_t> blk_val, val_words, post_dec;
  DevBuf<uint8_t> blk_voff;
  DevBuf<uint64_t> val_woff, poff_dec;
  DevBuf<ValSlice> blk_vs;
  uint64_t n_val_lists = 0, n_val_words = 0;
  std::vector<int> val_segs;        // which views are `_val` views
  std::vector<uint64_t> val_tbase;  // their first list
  ~SegList() {
    for (ii2_seg* g : v) delete g;
  }
};

// ---- ii2_merge over host buffers, pipelined by term range -----------------------------
// A compaction needs every segment, so H2D staging (PCIe) cannot overlap the kernels of the
// same terms.  It can overlap the kernels of OTHER terms: the term space is cut into P ranges
// at terms of the largest segment (host binary searches), every range is an independent
// compaction whose outputs concatenate (ranges are in term order), and the slices of range
// p+1 are uploaded on a second stream while range p is merged and its result flows back.
static int host_term_cmp(const uint8_t* a, uint32_t na, const uint8_t* b, uint32_t nb) {
  const int c = memcmp(a, b, na < nb ? na : nb);
  if (c) return c;
  return na < nb ? -1 : (na > nb ? 1 : 0);
}

// *bad is set when an offset pair met on the way is not inside [term_off[0], term_off[n]]
// (corrupt input: the caller falls back to the single-shot path, whose device-side check
// answers II2_ERR_INVALID); such a pair is never dereferenced.
static uint64_t host_lower_bound(const ii2_seg_view& v, const uint8_t* t, uint32_t nt, bool* bad) {
  uint64_t lo = 0, hi = v.n_terms;
  const uint32_t end = v.n_terms ? v.term_off[v.n_terms] : 0u;
  while (lo < hi) {
    const uint64_t mid = lo + ((hi - lo) >> 1);
    const uint32_t o = v.term_off[mid], e = v.term_off[mid + 1];
    if (e < o || e > end) {
      *bad = true;
      return lo;
    }
    const uint32_t n = e - o;
    if (host_term_cmp(v.term_bytes + o, n, t, nt) < 0)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

static int merge_single_shot(const ii2_seg_view* segs, int nseg, const uint32_t* removed_sorted,
                             uint64_t nrem, uint32_t flags, ii2_merge_out* out) {
  SegList list;
  for (int i = 0; i < nseg; i++) {
    ii2_seg* g = nullptr;
    II2_TRY(ii2_seg_upload(&segs[i], &g));
    list.v.push_back(g);
  }
  ii2_removed* rem = nullptr;
  if (nrem) II2_TRY(ii2_removed_upload(removed_sorted, nrem, &rem));
  std::unique_ptr<ii2_removed> rem_guard(rem);
  ii2_result* res = nullptr;
  II2_TRY(ii2_merge_dev(list.v.data(), nseg, rem,
                        II2_RESULT_ENCODED | ((flags & II2_MERGE_WANT_DECODED) ? II2_RESULT_DECODED : 0u),
                        &res));
  std::unique_ptr<ii2_result> res_guard(res);
  return ii2_result_download_merge(res, flags, out);
}

// internal: the pipelined path met input it leaves to the single-shot path (never returned)
constexpr int II2_ERR_RETRY_SINGLE = -1000;

struct EventList {
  std::vector<cudaEvent_t> v;
  ~EventList() {
    for (cudaEvent_t e : v) cudaEventDestroy(e);
  }
};

static int merge_pipelined(const ii2_seg_view* segs, int nseg, const uint32_t* removed_sorted,
                           uint64_t nrem, uint32_t flags, ii2_merge_out* out, int P,
                           std::unique_ptr<HostOwner>& own) {
  cudaStream_t sB = cur_stream(), sA = aux_stream();
  const bool want_dec = (flags & II2_MERGE_WANT_DECODED) != 0;
  // ---- range bounds: rows of nseg term indices, row 0 = starts, row P = ends
  int big = 0;
  for (int i = 1; i < nseg; i++)
    if (segs[i].n_terms > segs[big].n_terms) big = i;
  std::vector<uint64_t> bounds((size_t)(P + 1) * nseg, 0);
  uint64_t inst_total = 0;
  for (int i = 0; i < nseg; i++) {
    bounds[(size_t)P * nseg + i] = segs[i].n_terms;
    inst_total += segs[i].n_terms;
  }
  // The ranges are equal except the last two: what follows the last upload (its merge and the
  // download of its result) is the only part of the call the bus does not cover, so the last
  // range is small; 0.65 and 0.4 of a full range keep every range's merge + download shorter
  // than the next range's upload (measured on B200, C2: 30.1 instead of 30.5 ms per call).
  std::vector<double> cum(P + 1, 0.0);
  const bool taper = P >= 4 && segs[big].n_terms >= 64ull * P;
  for (int p = 0; p < P; p++)
    cum[p + 1] = cum[p] + (taper && p == P - 2 ? 0.65 : (taper && p == P - 1 ? 0.4 : 1.0));
  for (int p = 1; p < P; p++) {
    // equal ranges in integers (n_terms >= P: every cut is a different term, also when
    // n_terms == P); tapered ones are >= 25 terms apart
    const uint64_t at =
        taper ? std::min<uint64_t>(segs[big].n_terms - 1,
                                   (uint64_t)((double)segs[big].n_terms * (cum[p] / cum[P])))
              : segs[big].n_terms * (uint64_t)p / P;
    const uint32_t o = segs[big].term_off[at], e = segs[big].term_off[at + 1];
    if (e < o || e > segs[big].term_off[segs[big].n_terms]) return II2_ERR_RETRY_SINGLE;
    bool bad = false;
    for (int i = 0; i < nseg; i++)
      bounds[(size_t)p * nseg + i] =
          i == big ? at : host_lower_bound(segs[i], segs[big].term_bytes + o, e - o, &bad);
    if (bad) return II2_ERR_RETRY_SINGLE;
  }
  ii2_removed* rem = nullptr;
  if (nrem) II2_TRY(ii2_removed_upload(removed_sorted, nrem, &rem));
  std::unique_ptr<ii2_removed> rem_guard(rem);
  DevBuf<uint32_t> d_stats;
  II2_TRY(d_stats.alloc(2 * (size_t)P, sA));
  II2_CUDA_TRY(cudaMemsetAsync(d_stats.p, 0, 8 * (size_t)P, sA));
  EventList ev;
  for (int p = 0; p < P; p++) {
    cudaEvent_t e;
    II2_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ev.v.push_back(e);
  }
  std::vector<std::unique_ptr<SegList>> parts(P);
  std::vector<std::unique_ptr<ii2_result>> results(P);
  // Are the caller's arrays pinned and visible to the device (unified addressing)?  Then a
  // kernel gathers them (k_gather_host); pageable arrays go through the copy engine.  (A
  // copy-engine request per slice was measured slower on pinned inputs too, on B200: 36.8 vs
  // 31.1 ms per C2 call, on one to four streams — the fixed cost of a request does not overlap.)
  struct DevAlias {
    const uint8_t* tb;
    const uint8_t* toff;
    const uint8_t* post;  // DECODED: postings; `_val` view: the `_val` bytes
    const uint8_t* poff;  // DECODED: posting offsets; `_val` view: the FST outputs
  };
  auto is_val = [&](int i) { return segs[i].mode == II2_SEG_VAL; };
  // FST output of term t of a `_val` view in bytes (t == n_terms: the end of the file)
  auto val_at = [&](const ii2_seg_view& v, uint64_t t) -> uint64_t {
    if (t >= v.n_terms) return v.val_size;
    return v.val_woff32 ? 4ull * v.val_woff32[t] : v.val_off[t];
  };
  std::vector<DevAlias> alias(nseg);
  bool gather = true;
  auto dev_alias = [&](const void* hp, size_t align, const uint8_t** out_p) {
    *out_p = nullptr;
    if (!hp) return;  // empty array: nothing to read
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, hp) != cudaSuccess) {
      cudaGetLastError();
      gather = false;
      return;
    }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer ||
        (reinterpret_cast<uintptr_t>(at.devicePointer) & (align - 1)) !=
            (reinterpret_cast<uintptr_t>(hp) & (align - 1)) ||
        (reinterpret_cast<uintptr_t>(hp) & (align - 1)) != 0) {
      gather = false;
      return;
    }
    *out_p = static_cast<const uint8_t*>(at.devicePointer);
  };
  for (int i = 0; i < nseg && gather; i++) {
    dev_alias(segs[i].term_bytes, 4, &alias[i].tb);
    dev_alias(segs[i].term_off, 4, &alias[i].toff);
    if (is_val(i)) {
      dev_alias(segs[i].val_bytes, 4, &alias[i].post);
      if (segs[i].val_woff32)
        dev_alias(segs[i].val_woff32, 4, &alias[i].poff);
      else
        dev_alias(segs[i].val_off, 8, &alias[i].poff);
    } else {
      dev_alias(segs[i].post, 4, &alias[i].post);
      dev_alias(segs[i].post_off, 8, &alias[i].poff);
    }
  }

  // Stage the slices of range p: four allocations and one check launch for all segments (an
  // allocation + a kernel per slice would cost more host time than the copies take).  Offsets
  // stay absolute: the slice's base pointers are moved back by its first offset instead.  Every
  // slice lands at the same phase modulo 512 bytes as its source (vector copies; the moved term
  // pointer keeps the 4-byte alignment the key loads need).
  const size_t nx = (size_t)nseg;
  const size_t ref_bytes = (sizeof(SliceRef) * nx + 15) & ~(size_t)15;
  const size_t job_bytes = sizeof(GatherJob) * 4 * nx;
  PinnedBlock tab_blk((ref_bytes + job_bytes) * P);
  uint8_t* h_tab = static_cast<uint8_t*>(tab_blk.p);
  if (!h_tab) return II2_ERR_NOMEM;
  PinnedBlock vtab_blk(sizeof(ValSlice) * nx * P + 64);
  uint8_t* h_vtab = static_cast<uint8_t*>(vtab_blk.p);
  if (!h_vtab) return II2_ERR_NOMEM;
  auto enqueue_upload = [&](int p) -> int {
    parts[p].reset(new SegList());
    SegList& L = *parts[p];
    const uint64_t* lo = &bounds[(size_t)p * nseg];
    const uint64_t* hi = &bounds[(size_t)(p + 1) * nseg];
    size_t tb_bytes = 0, toff_bytes = 0, post_bytes = 0, poff_bytes = 0, val_bytes = 0, voff_bytes = 0;
    uint64_t val_lists = 0, val_words = 0;
    int n_val = 0;
    for (int i = 0; i < nseg; i++) {
      const ii2_seg_view& v = segs[i];
      // corrupt offsets are II2_ERR_INVALID, like on the single-shot path, before any size is
      // computed from a wrapped difference
      if (hi[i] < lo[i] || v.term_off[hi[i]] < v.term_off[lo[i]]) return II2_ERR_INVALID;
      const size_t n1 = (size_t)(hi[i] - lo[i]) + 1;
      // every slice: up to 2 x 511 bytes of phase (placed at its source's phase modulo 512)
      tb_bytes += (size_t)(v.term_off[hi[i]] - v.term_off[lo[i]]) + 2 * kGatherAlign + 64;  // + tail padding
      toff_bytes += n1 * 4 + 2 * kGatherAlign;
      if (is_val(i)) {
        const uint64_t b0 = val_at(v, lo[i]), b1 = val_at(v, hi[i]);
        if (b1 < b0 || b1 > v.val_size || ((b0 | b1) & 3)) return II2_ERR_INVALID;
        val_bytes += (size_t)(b1 - b0) + 2 * kGatherAlign;
        voff_bytes += n1 * 8 + 2 * kGatherAlign;
        val_lists += hi[i] - lo[i];
        val_words += (b1 - b0) / 4;
        n_val++;
      } else {
        if (v.post_off[hi[i]] < v.post_off[lo[i]]) return II2_ERR_INVALID;
        post_bytes += (size_t)(v.post_off[hi[i]] - v.post_off[lo[i]]) * 4 + 2 * kGatherAlign;
        poff_bytes += n1 * 8 + 2 * kGatherAlign;
      }
    }
    II2_TRY(L.blk_tb.alloc(tb_bytes, sA, 64));
    II2_TRY(L.blk_toff.alloc(toff_bytes / 4, sA));
    II2_TRY(L.blk_post.alloc(post_bytes / 4, sA, 16));
    II2_TRY(L.blk_poff.alloc(poff_bytes / 8, sA));
    II2_TRY(L.blk_ref.alloc(nx, sA));
    L.n_val_lists = val_lists;
    L.n_val_words = val_words;
    std::vector<ValSlice> h_vs;
    if (n_val) {
      II2_TRY(L.blk_val.alloc(val_bytes / 4, sA, 16));
      II2_TRY(L.blk_voff.alloc(voff_bytes, sA, 16));
      II2_TRY(L.val_words.alloc(val_words, sA, 64));
      II2_TRY(L.val_woff.alloc(val_lists + 1, sA));
      II2_TRY(L.blk_vs.alloc(n_val, sA));
    }
    size_t at_val = 0, at_voff = 0;
    uint64_t run_lists = 0, run_words = 0;
    if (gather) II2_TRY(L.blk_job.alloc(4 * nx, sA));
    SliceRef* refs = reinterpret_cast<SliceRef*>(h_tab + (ref_bytes + job_bytes) * p);
    GatherJob* jobs = reinterpret_cast<GatherJob*>(h_tab + (ref_bytes + job_bytes) * p + ref_bytes);
    uint32_t njobs = 0;
    uint64_t nvec = 0;
    size_t at_tb = 0, at_toff = 0, at_post = 0, at_poff = 0;  // byte cursors
    uint32_t max_n = 0;
    // one array slice: place it at the phase of its source, queue its copy
    // `first` = the slice's first offset inside its array, in bytes.  The gather kernel needs
    // dst = src (mod 512); a copy engine does not, and then the slice lands at the phase of
    // `first`, so that the moved base pointer (dst - first) is 512-byte aligned whatever the
    // alignment of the caller's pointer (a Go sub-slice or an mmap offset may start anywhere;
    // the key loads need a 4-byte aligned term base).
    auto place = [&](uint8_t* blk, size_t& cursor, const void* hsrc, const uint8_t* dsrc,
                     uint64_t bytes, uint64_t first, uint8_t** dst_out) -> int {
      const uint8_t* src = gather ? dsrc : static_cast<const uint8_t*>(hsrc);
      cursor = ((cursor + kGatherAlign - 1) & ~(size_t)(kGatherAlign - 1)) +
               (gather ? (reinterpret_cast<uintptr_t>(src) & (kGatherAlign - 1))
                       : (size_t)(first & (kGatherAlign - 1)));
      uint8_t* dst = blk + cursor;
      *dst_out = dst;
      cursor += bytes;
      if (!bytes) return II2_OK;
      if (gather) {
        GatherJob& g = jobs[njobs++];
        g.src = src;
        g.dst = dst;
        g.bytes = bytes;
        g.vec0 = nvec;
        nvec += gather_job_vectors(src, bytes);
      } else {
        II2_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, sA));
      }
      return II2_OK;
    };
    for (int i = 0; i < nseg; i++) {
      const ii2_seg_view& v = segs[i];
      const uint64_t n = hi[i] - lo[i];
      const uint32_t tfirst = v.term_off[lo[i]];
      const uint64_t tlen = v.term_off[hi[i]] - tfirst;
      if (tlen && !v.term_bytes) return II2_ERR_INVALID;
      uint8_t *d_tb, *d_toff, *d_post = nullptr, *d_poff = nullptr;
      II2_TRY(place(L.blk_tb.p, at_tb, v.term_bytes ? v.term_bytes + tfirst : nullptr,
                    alias[i].tb ? alias[i].tb + tfirst : nullptr, tlen, tfirst, &d_tb));
      at_tb += 32;  // key loads read past the last term
      II2_TRY(place(reinterpret_cast<uint8_t*>(L.blk_toff.p), at_toff, v.term_off + lo[i],
                    alias[i].toff + 4 * lo[i], (n + 1) * 4, 4 * lo[i], &d_toff));
      std::unique_ptr<ii2_seg> g(new ii2_seg());
      g->n_terms = (uint32_t)n;
      g->term_bytes_len = tlen;
      // non-owning views into the blocks (scratch = true: never freed through the view)
      g->tb.p = d_tb - tfirst;
      g->tb.scratch = true;
      g->toff.p = reinterpret_cast<uint32_t*>(d_toff);
      g->toff.scratch = true;
      g->post.scratch = true;
      g->poff.scratch = true;
      if (is_val(i)) {
        // the `_val` run of the slice and the FST outputs of its terms; post / poff of the view
        // are filled in once the range has been decoded (finish_val)
        const uint64_t b0 = val_at(v, lo[i]), b1 = val_at(v, hi[i]);
        uint8_t *d_val, *d_vo;
        II2_TRY(place(reinterpret_cast<uint8_t*>(L.blk_val.p), at_val, v.val_bytes + b0,
                      alias[i].post ? alias[i].post + b0 : nullptr, b1 - b0, b0, &d_val));
        const bool w32 = v.val_woff32 != nullptr;
        const size_t esz = w32 ? 4 : 8;
        II2_TRY(place(L.blk_voff.p, at_voff,
                      w32 ? static_cast<const void*>(v.val_woff32 + lo[i]) : static_cast<const void*>(v.val_off + lo[i]),
                      alias[i].poff ? alias[i].poff + esz * lo[i] : nullptr, n * esz, esz * lo[i], &d_vo));
        ValSlice vs;
        vs.src = reinterpret_cast<const uint32_t*>(d_val);
        vs.off = d_vo;
        vs.first = b0;
        vs.words = (b1 - b0) / 4;
        vs.wbase = run_words;
        vs.tbase = run_lists;
        vs.n = (uint32_t)n;
        vs.off32 = w32 ? 1u : 0u;
        h_vs.push_back(vs);
        L.val_segs.push_back(i);
        L.val_tbase.push_back(run_lists);
        run_words += vs.words;
        run_lists += n;
        g->n_post = 0;
      } else {
        const uint64_t pfirst = v.post_off[lo[i]], plen = v.post_off[hi[i]] - pfirst;
        if (plen && !v.post) return II2_ERR_INVALID;
        II2_TRY(place(reinterpret_cast<uint8_t*>(L.blk_post.p), at_post, v.post ? v.post + pfirst : nullptr,
                      alias[i].post ? alias[i].post + 4 * pfirst : nullptr, plen * 4, 4 * pfirst, &d_post));
        II2_TRY(place(reinterpret_cast<uint8_t*>(L.blk_poff.p), at_poff, v.post_off + lo[i],
                      alias[i].poff + 8 * lo[i], (n + 1) * 8, 8 * lo[i], &d_poff));
        g->n_post = plen;
        g->post.p = reinterpret_cast<uint32_t*>(d_post) - pfirst;
        g->poff.p = reinterpret_cast<uint64_t*>(d_poff);
      }
      refs[i].toff = g->toff.p;
      refs[i].poff = g->poff.p;  // null for a `_val` view: its posting offsets come from the decoder
      refs[i].n = (uint32_t)n;
      refs[i].pad = 0;
      max_n = std::max<uint32_t>(max_n, (uint32_t)n);
      L.v.push_back(g.release());
    }
    II2_TRY(small_copy(L.blk_ref.p, refs, sizeof(SliceRef) * nx, sA));
    if (gather && njobs) {
      II2_TRY(small_copy(L.blk_job.p, jobs, sizeof(GatherJob) * njobs, sA));
      // at most 64 CTAs: the staging kernel shares the SMs with the merge (32 and 128 were
      // measured no faster)
      const unsigned grid = (unsigned)std::min<uint64_t>(
          64, std::max<uint64_t>(1, div_up(nvec, (uint64_t)kGatherThreads * kGatherUnroll)));
      k_gather_host<<<grid, kGatherThreads, 0, sA>>>(L.blk_job.p, njobs, nvec);
      II2_LAUNCHED();
    }
    if (max_n) {
      const dim3 grid(std::min<unsigned>(div_up(max_n, 256), 64u), (unsigned)nseg);
      k_slices_check<<<grid, 256, 0, sA>>>(L.blk_ref.p, d_stats.p + 2 * p);
      II2_LAUNCHED();
    }
    if (!h_vs.empty()) {  // `_val` slices back to back + the word offset of every list
      ValSlice* h_tab_vs = reinterpret_cast<ValSlice*>(h_vtab + (size_t)p * nx * sizeof(ValSlice));
      memcpy(h_tab_vs, h_vs.data(), h_vs.size() * sizeof(ValSlice));
      II2_TRY(small_copy(L.blk_vs.p, h_tab_vs, h_vs.size() * sizeof(ValSlice), sA));
      uint64_t max_w = 0;
      uint32_t max_t = 0;
      for (const ValSlice& x : h_vs) {
        max_w = std::max(max_w, x.words);
        max_t = std::max(max_t, x.n);
      }
      const unsigned ns = (unsigned)h_vs.size();
      if (max_w) {
        k_val_compact<<<dim3(std::min<unsigned>(div_up(max_w, 256), 256u), ns), 256, 0, sA>>>(L.blk_vs.p, L.val_words.p);
        II2_LAUNCHED();
      }
      k_val_woff<<<dim3(std::max(1u, std::min<unsigned>(div_up(max_t, 256), 64u)), ns), 256, 0, sA>>>(
          L.blk_vs.p, ns, L.val_woff.p, d_stats.p + 2 * p);
      II2_LAUNCHED();
    }
    II2_CUDA_TRY(cudaEventRecord(ev.v[p], sA));
    return II2_OK;
  };

  // ---- output buffers: sized from the first range's result, exact re-copy if that was short
  own.reset(new HostOwner());
  uint64_t capT = 0, capTB = 0, capE = 0, capP = 0;
  uint64_t runT = 0, runTB = 0, runE = 0, runP = 0;
  bool overflow = false;
  uint64_t terms_merged = 0, postings_in = 0;
  std::string min_term, max_term;
  bool has_minmax = false;
  auto alloc_out = [&](uint64_t T, uint64_t TB, uint64_t E, uint64_t Pn) -> int {
    own.reset(new HostOwner());
    out->term_bytes = own->alloc<uint8_t>(TB);
    out->term_off = own->alloc<uint32_t>(T + 1);
    out->val_off = own->alloc<uint64_t>(T);
    out->val_bytes = reinterpret_cast<uint8_t*>(own->alloc<uint32_t>(E));
    if (!out->term_bytes || !out->term_off || !out->val_off || !out->val_bytes) return II2_ERR_NOMEM;
    if (want_dec) {
      out->post = own->alloc<uint32_t>(Pn);
      out->post_off = own->alloc<uint64_t>(T + 1);
      if (!out->post || !out->post_off) return II2_ERR_NOMEM;
    }
    capT = T; capTB = TB; capE = E; capP = Pn;
    return II2_OK;
  };
  // copies result r to the output at the running offsets (offset arrays get their base added
  // on the device first, once)
  auto copy_out = [&](ii2_result* r, uint64_t bT, uint64_t bTB, uint64_t bE, uint64_t bP,
                      bool rebase) -> int {
    if (rebase && r->T) {
      if (bTB) {
        k_rebase_u32<<<div_up(r->T, 256), 256, 0, sB>>>(r->out.term_off.p, r->T, (uint32_t)(0u - (uint32_t)bTB));
        II2_LAUNCHED();
      }
      if (bE) {
        k_rebase_u64<<<div_up(r->T, 256), 256, 0, sB>>>(r->out.val_off.p, r->T, 0ull - 4ull * bE);
        II2_LAUNCHED();
      }
      if (want_dec && bP) {
        k_rebase_u64<<<div_up(r->T, 256), 256, 0, sB>>>(r->out.post_off.p, r->T, 0ull - bP);
        II2_LAUNCHED();
      }
    }
    if (r->TB)
      II2_CUDA_TRY(cudaMemcpyAsync(out->term_bytes + bTB, r->out.term_bytes.p, r->TB, cudaMemcpyDeviceToHost, sB));
    if (r->T) {
      II2_CUDA_TRY(cudaMemcpyAsync(out->term_off + bT, r->out.term_off.p, r->T * 4, cudaMemcpyDeviceToHost, sB));
      II2_CUDA_TRY(cudaMemcpyAsync(out->val_off + bT, r->out.val_off.p, r->T * 8, cudaMemcpyDeviceToHost, sB));
    }
    if (r->E)
      II2_CUDA_TRY(cudaMemcpyAsync(out->val_bytes + 4 * bE, r->out.val_words.p, r->E * 4, cudaMemcpyDeviceToHost, sB));
    if (want_dec) {
      if (r->P)
        II2_CUDA_TRY(cudaMemcpyAsync(out->post + bP, r->out.post.p, r->P * 4, cudaMemcpyDeviceToHost, sB));
      if (r->T)
        II2_CUDA_TRY(cudaMemcpyAsync(out->post_off + bT, r->out.post_off.p, r->T * 8, cudaMemcpyDeviceToHost, sB));
    }
    return II2_OK;
  };

  {  // range 0 crosses the bus alone; the later ranges share it with kernels and downloads
    ProfScope sc("e2e_upload_first", sA);
    II2_TRY(enqueue_upload(0));
  }
  for (int p = 0; p < P; p++) {
    if (p + 1 < P) {  // in flight while range p is merged
      ProfScope sc("e2e_enqueue_upload", sA);
      II2_TRY(enqueue_upload(p + 1));
    }
    II2_CUDA_TRY(cudaStreamWaitEvent(sB, ev.v[p], 0));
    {
      ProfScope sc("e2e_wait_upload", sB);
      II2_TRY(seg_check_result(d_stats.p + 2 * p, sB));
    }
    if (parts[p]->n_val_lists) {  // the `_val` views of the range: one batched decode (K3a)
      SegList& L = *parts[p];
      ProfScope sc("e2e_val_decode", sB);
      uint64_t total = 0;
      II2_TRY(intcomp_decode_dev(L.val_words.p, L.val_woff.p, L.n_val_lists, L.post_dec, L.poff_dec,
                                 &total, sB, false));
      arena_reset(sB);  // (the decoder's temporaries; its outputs are stream-ordered allocations)
      for (size_t j = 0; j < L.val_segs.size(); j++) {
        ii2_seg* g = L.v[L.val_segs[j]];
        g->post.p = L.post_dec.p;                       // offsets index the shared decoded array
        g->poff.p = L.poff_dec.p + L.val_tbase[j];
        g->n_post = j == 0 ? total : 0;                 // (only the sum over the views is used)
      }
    }
    ii2_result* res = nullptr;
    II2_TRY(run_pipeline(parts[p]->v.data(), nseg, nullptr, 0, false, nullptr, 0, false, rem,
                         want_dec, true, true, false, &res));
    results[p].reset(res);
    parts[p].reset();  // the stream is drained: the slices can go
    terms_merged += res->terms_merged;
    postings_in += res->postings_in;
    if (res->has_minmax) {
      if (!has_minmax) min_term = res->min_term;
      max_term = res->max_term;
      has_minmax = true;
    }
    if (p == 0) {  // extrapolate by instances, a quarter of slack
      uint64_t inst0 = 0;
      for (int i = 0; i < nseg; i++) inst0 += bounds[(size_t)nseg + i];
      // II2_MERGE_SLACK=<x> replaces the 1.25 (tests: a small value forces the exact re-copy)
      const char* env_slack = getenv("II2_MERGE_SLACK");
      const double slack = env_slack ? atof(env_slack) : 1.25;
      const double f = inst0 ? slack * (double)inst_total / (double)inst0 : (double)P;
      II2_TRY(alloc_out((uint64_t)(res->T * f) + 4096, (uint64_t)(res->TB * f) + 65536,
                        (uint64_t)(res->E * f) + 65536, want_dec ? (uint64_t)(res->P * f) + 65536 : 0));
    }
    if (runT + res->T > capT || runTB + res->TB > capTB || runE + res->E > capE ||
        (want_dec && runP + res->P > capP))
      overflow = true;
    if (!overflow) {
      ProfScope sc("e2e_enqueue_download", sB);
      II2_TRY(copy_out(res, runT, runTB, runE, runP, true));
      res->rebased = true;
    }
    runT += res->T;
    runTB += res->TB;
    runE += res->E;
    runP += res->P;
    if (runTB >= (1ull << 32)) {
      set_last_error("merged term dictionary exceeds 4 GiB of term bytes");
      return II2_ERR_UNSUPPORTED;
    }
  }
  if (overflow) {  // the estimate was short: exact buffers, copy every range again
    II2_CUDA_TRY(cudaStreamSynchronize(sB));
    II2_TRY(alloc_out(runT, runTB, runE, want_dec ? runP : 0));
    uint64_t bT = 0, bTB = 0, bE = 0, bP = 0;
    for (int p = 0; p < P; p++) {
      ii2_result* r = results[p].get();
      II2_TRY(copy_out(r, bT, bTB, bE, bP, !r->rebased));  // same bases as in the first pass
      r->rebased = true;
      bT += r->T;
      bTB += r->TB;
      bE += r->E;
      bP += r->P;
    }
  }
  {
    ProfScope sc("e2e_final_sync", sB);
    II2_CUDA_TRY(cudaStreamSynchronize(sB));
  }
  out->term_off[runT] = (uint32_t)runTB;
  if (want_dec) out->post_off[runT] = runP;
  out->terms_count = runT;
  out->val_size = runE * 4;
  out->has_minmax = has_minmax ? 1 : 0;
  if (has_minmax) {
    out->min_term = own->alloc<uint8_t>(min_term.size() + 1);
    out->max_term = own->alloc<uint8_t>(max_term.size() + 1);
    if (!out->min_term || !out->max_term) return II2_ERR_NOMEM;
    memcpy(out->min_term, min_term.data(), min_term.size());
    memcpy(out->max_term, max_term.data(), max_term.size());
    out->min_term_len = (uint32_t)min_term.size();
    out->max_term_len = (uint32_t)max_term.size();
  }
  out->terms_merged = terms_merged;
  out->postings_in = postings_in;
  out->postings_out = runP;
  out->_owner = own.release();
  return II2_OK;
}

int ii2_merge(const ii2_seg_view* segs, int nseg, const uint32_t* removed_sorted, uint64_t nrem,
              uint32_t flags, ii2_merge_out* out) {
  if (!out || nseg < 0 || (nseg && !segs)) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  II2_TRY(ctx_require());
  // term-range pipelining pays once staging dominates: DECODED views (no per-segment host
  // synchronisation), at least ~200 MB per range
  // (DECODED views and `_val` views — what a Go caller holds: the mmap of <key>_val and the FST
  // outputs, file/reader.go:50-52,79-100 — are staged per term range; DIRECT views are tiny)
  uint64_t bytes = 0;
  bool all_decoded = nseg > 0;
  for (int i = 0; i < nseg; i++) {
    const ii2_seg_view& v = segs[i];
    // (an empty segment may come with NULL arrays: the pipelined path indexes them, the
    // single-shot path does not)
    const bool dec = v.mode == II2_SEG_DECODED && v.term_off && v.post_off;
    const bool val = v.mode == II2_SEG_VAL && v.term_off && (v.val_off || v.val_woff32) && v.n_terms &&
                     !(v.val_size & 3) && (v.val_size || !v.n_terms) && v.val_bytes;
    if (!dec && !val) {
      all_decoded = false;
      break;
    }
    if (v.n_terms)
      bytes += (uint64_t)(v.term_off[v.n_terms] - v.term_off[0]) + 4ull * v.n_terms +
               (dec ? 8ull * v.n_terms + 4ull * (v.post_off[v.n_terms] - v.post_off[0])
                    : (v.val_woff32 ? 4ull : 8ull) * v.n_terms + v.val_size);
  }
  // II2_MERGE_PARTS=<n> forces the number of ranges (tests and tuning; 1 = single shot)
  const char* env_parts = getenv("II2_MERGE_PARTS");
  const int forced = env_parts ? atoi(env_parts) : 0;
  // measured on B200 (1.25 GB of inputs): 35.6 ms single shot, 31.1 ms with 6 ranges, 32.1 with 8
  int P = forced > 0 ? forced : (int)std::min<uint64_t>(6, bytes / (192ull << 20));
  if (!all_decoded || P < 2) return merge_single_shot(segs, nseg, removed_sorted, nrem, flags, out);
  uint64_t max_terms = 0;
  for (int i = 0; i < nseg; i++) max_terms = std::max<uint64_t>(max_terms, segs[i].n_terms);
  if (max_terms < (uint64_t)P) return merge_single_shot(segs, nseg, removed_sorted, nrem, flags, out);
  std::unique_ptr<HostOwner> own;  // outlives any copy still in flight when a step fails
  int rc = merge_pipelined(segs, nseg, removed_sorted, nrem, flags, out, P, own);
  if (rc == II2_ERR_RETRY_SINGLE) {  // nothing was enqueued yet
    memset(out, 0, sizeof(*out));
    return merge_single_shot(segs, nseg, removed_sorted, nrem, flags, out);
  }
  if (rc != II2_OK) {
    cudaStreamSynchronize(cur_stream());
    cudaStreamSynchronize(aux_stream());
    memset(out, 0, sizeof(*out));
  }
  return rc;
}

int ii2_read_range(const ii2_seg_view* segs, int nseg, const uint8_t* min, size_t minlen,
                   const uint8_t* max, size_t maxlen, const uint32_t* removed_sorted,
                   uint64_t nrem, ii2_read_out* out) {
  if (!out || nseg < 0 || (nseg && !segs)) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  II2_TRY(ctx_require());
  SegList list;
  for (int i = 0; i < nseg; i++) {
    ii2_seg* g = nullptr;
    II2_TRY(ii2_seg_upload(&segs[i], &g));
    list.v.push_back(g);
  }
  ii2_removed* rem = nullptr;
  if (removed_sorted) II2_TRY(ii2_removed_upload(removed_sorted, nrem, &rem));
  std::unique_ptr<ii2_removed> rem_guard(rem);
  ii2_result* res = nullptr;
  II2_TRY(ii2_read_range_dev(list.v.data(), nseg, min, minlen, max, maxlen, rem, &res));
  std::unique_ptr<ii2_result> res_guard(res);
  return ii2_result_download_read(res, out);
}

int ii2_prefix_search(const ii2_seg_view* segs, int nseg, const uint8_t* prefix_bytes,
                      const uint32_t* prefix_off, uint32_t nprefix, ii2_prefix_out* out) {
  if (!out || nseg < 0 || (nseg && !segs)) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  II2_TRY(ctx_require());
  SegList list;
  for (int i = 0; i < nseg; i++) {
    ii2_seg* g = nullptr;
    II2_TRY(ii2_seg_upload(&segs[i], &g));
    list.v.push_back(g);
  }
  return ii2_prefix_search_dev(list.v.data(), nseg, prefix_bytes, prefix_off, nprefix, out);
}

int ii2_lookup(const ii2_seg_view* segs, int nseg, const uint8_t* key_bytes,
               const uint32_t* key_off, uint32_t nkeys, const uint32_t* removed_sorted,
               uint64_t nrem, ii2_lookup_out* out) {
  if (!out || nseg < 0 || (nseg && !segs) || (nkeys && !key_off)) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  II2_TRY(ctx_require());
  SegList list;
  for (int i = 0; i < nseg; i++) {
    ii2_seg* g = nullptr;
    II2_TRY(ii2_seg_upload(&segs[i], &g));
    list.v.push_back(g);
  }
  ii2_removed* rem = nullptr;
  if (removed_sorted) II2_TRY(ii2_removed_upload(removed_sorted, nrem, &rem));
  std::unique_ptr<ii2_removed> rem_guard(rem);
  return ii2_lookup_dev(list.v.data(), nseg, key_bytes, key_off, nkeys, rem, out);
}

int ii2_query(const ii2_seg_view* segs, int nseg, const ii2_query_batch* q,
              const uint32_t* removed_sorted, uint64_t nrem, ii2_query_out* out) {
  if (!out) return II2_ERR_INVALID;
  memset(out, 0, sizeof(*out));
  if (!q || nseg < 0 || (nseg && !segs)) return II2_ERR_INVALID;
  II2_TRY(ctx_require());
  SegList list;
  for (int i = 0; i < nseg; i++) {
    ii2_seg* g = nullptr;
    II2_TRY(ii2_seg_upload(&segs[i], &g));
    list.v.push_back(g);
  }
  ii2_removed* rem = nullptr;
  if (removed_sorted) II2_TRY(ii2_removed_upload(removed_sorted, nrem, &rem));
  std::unique_ptr<ii2_removed> rem_guard(rem);
  return ii2_query_dev(list.v.data(), nseg, q, rem, out);
}

}  // extern "C"
