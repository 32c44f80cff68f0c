// k8_lookup.cu — K8: Read(t, t) for a batch of keys t in one call (ii2_lookup_dev).
//
// A single point read (k12_union.cu, k4_point_kernel) is one kernel and still costs ~60 us:
// launch, host round trip and the kernel's dependent chain, not bytes.  A caller with N keys
// (the terms of a query, the point reads of many goroutines) paid N of those.  Here the whole
// batch is a fixed number of launches and two host synchronisations (one to size the output,
// one for the copy back):
//   k8_lookup_kernel  one CTA per key (grid-stride): the 8 warps search the segments (the
//                     32-way exact search of the point read), the segments that hold the key
//                     are compacted in segment order with block scans, and a key of at most
//                     4096 values is unioned in shared memory by cta_union_term<8> — single
//                     source passed through as stored (survey Q4), otherwise sorted-unique,
//                     removed filter by bitmap or sorted list.  The union lands in an output
//                     pool by bump allocation; the pool holds min(nkeys * 4096, Σ postings of
//                     the segments) values, which every batch of distinct keys fits.
//   deferred keys     more than 4096 values, or a union the pool could not take (repeated keys):
//                     their sources are found again (k8_sources_kernel) and the multi-CTA heavy
//                     union runs on them (k2_large_run, single sources passed through).  Rare;
//                     host round trips are acceptable there.
//   placement         exact per-key counts -> exclusive scan -> k8_place copies the lists back
//                     to back.
#include <algorithm>
#include <vector>

#include "lookup.cuh"
#include "union_dev.cuh"

namespace ii2 {

namespace {

constexpr uint32_t kLookupCap = 8 * MED_RUN;  // 4096 values: what cta_union_term<8> unions
constexpr uint32_t kKeyStage = (kLookupCap + kLookupCap / 16) * 4;  // key bytes staged in s_o

struct K8Args {
  const SegDesc* segs;
  int k;
  const uint8_t* kb;
  const uint32_t* koff;  // [nkeys + 1]
  uint32_t nkeys;
  RemovedSet rem;
  int keep_empty;
  uint8_t* found;        // [nkeys]
  uint64_t* cnt;         // [nkeys + 1] values of key i (their exclusive scan is post_off)
  uint64_t* ptr;         // [nkeys] device address of key i's values
  uint32_t* pool;
  uint64_t pool_cap;
  unsigned long long* ctr;  // [0] pool cursor, [1] deferred keys, [2] postings in
  uint32_t* def_key;     // [nkeys] deferred keys
  uint32_t* def_c;       // [nkeys] and the number of segments that hold each
};

// Looks key (kp, kn) up in every segment; the segments that hold it are handed, in segment
// order, to emit(j, address of the list, its length, Σ lengths before it).  Returns their count
// c and their total length in L.  Every thread of the 256-thread CTA calls.  Warp w searches
// the segments base + 32 w + j one after the other; lane j keeps the answer for segment
// base + 32 w + j, so thread t holds segment base + t for the block scans.
template <class Emit>
__device__ __forceinline__ uint32_t find_sources(const SegDesc* __restrict__ segs, int k,
                                                 const uint8_t* kp, uint32_t kn, uint64_t& L,
                                                 uint64_t* s_ws, uint32_t* s_ws32, Emit emit) {
  const uint32_t lane = lane_id(), w = warp_id();
  uint32_t c = 0;
  uint64_t run = 0;
  for (int base = 0; base < k; base += 256) {
    uint64_t my_ptr = 0, my_len = 0;
    bool my_present = false;
    for (int j = 0; j < 32; j++) {
      const int s = base + (int)w * 32 + j;
      if (s >= k) break;  // uniform inside the warp
      const SegDesc sd = segs[s];
      auto term_vs = [&](uint32_t i) {
        const uint32_t o = __ldg(sd.toff + i), n = __ldg(sd.toff + i + 1) - o;
        return term_compare(sd.tb + o, n, kp, kn);
      };
      const uint32_t lo = warp_partition_point(0u, sd.n, [&](uint32_t i) { return term_vs(i) < 0; });
      const bool hit = lo < sd.n && term_vs(lo) == 0;
      if (hit && lane == (uint32_t)j) {
        const uint64_t p0 = __ldg(sd.poff + lo), p1 = __ldg(sd.poff + lo + 1);
        my_present = true;
        my_ptr = reinterpret_cast<uint64_t>(sd.post + p0);
        my_len = p1 - p0;
      }
    }
    uint32_t ctot;
    uint64_t ltot;
    const uint32_t ex_c = block_exclusive_scan<uint32_t>(my_present ? 1u : 0u, s_ws32, ctot);
    const uint64_t ex_l = block_exclusive_scan<uint64_t>(my_len, s_ws, ltot);
    if (my_present) emit(c + ex_c, my_ptr, my_len, run + ex_l);
    c += ctot;
    run += ltot;
  }
  L = run;
  return c;
}

__global__ void __launch_bounds__(256) k8_lookup_kernel(const K8Args a) {
  __shared__ uint32_t s_v[kLookupCap];  // sources of the key (u64), then the union's survivors
  __shared__ uint32_t s_o[kLookupCap + kLookupCap / 16];  // the key's bytes, then the gather
  __shared__ uint32_t s_moff[kMaxSegs + 1];
  __shared__ uint64_t s_ws[256 / 32 + 2];
  __shared__ uint32_t s_ws32[256 / 32 + 2];
  __shared__ uint32_t s_cnt[8], s_last[8];
  __shared__ unsigned long long s_pos;
  // The compacted source pointers live in s_v: cta_union_term reads them from there (its copy
  // into s_v is then in place) and writes s_v only after barriers that follow every read.
  uint64_t* const s_src = reinterpret_cast<uint64_t*>(s_v);
  uint8_t* const s_key = reinterpret_cast<uint8_t*>(s_o);
  const uint32_t tid = threadIdx.x;
  for (uint32_t i = blockIdx.x; i < a.nkeys; i += gridDim.x) {
    const uint32_t k0 = a.koff[i], kn = a.koff[i + 1] - k0;
    const uint8_t* kp = a.kb + k0;
    __syncthreads();  // the previous key is done with s_v / s_o / s_moff
    if (kn <= kKeyStage) {  // uniform
      for (uint32_t t = tid; t < kn; t += 256) s_key[t] = kp[t];
      kp = s_key;
      __syncthreads();
    }
    uint64_t L;
    const uint32_t c = find_sources(a.segs, a.k, kp, kn, L, s_ws, s_ws32,
                                    [&](uint32_t j, uint64_t p, uint64_t, uint64_t before) {
                                      s_src[j] = p;
                                      s_moff[j] = (uint32_t)min(before, (uint64_t)kLookupCap + 1);
                                    });
    if (tid == 0) {
      s_moff[c] = (uint32_t)min(L, (uint64_t)kLookupCap + 1);
      if (L) atomicAdd(&a.ctr[2], (unsigned long long)L);
    }
    __syncthreads();
    bool defer = false;
    if (c == 0) {  // uniform
      if (tid == 0) {
        a.found[i] = 0;
        a.cnt[i] = 0;
        a.ptr[i] = 0;
      }
      continue;
    }
    if (L <= kLookupCap) {  // uniform
      const uint32_t outn = cta_union_term<8>(s_src, c, (uint32_t)L, a.rem, s_v, s_o, s_moff, s_cnt, s_last);
      if (tid == 0) s_pos = atomicAdd(&a.ctr[0], (unsigned long long)outn);
      __syncthreads();
      const uint64_t pos = s_pos;
      if (outn == 0 || pos + outn <= a.pool_cap) {
        uint32_t* const dst = a.pool + pos;
        for (uint32_t e = tid; e < outn; e += 256) dst[e] = s_v[e];
        if (tid == 0) {
          a.found[i] = (outn || a.keep_empty) ? 1 : 0;
          a.cnt[i] = outn;
          a.ptr[i] = reinterpret_cast<uint64_t>(dst);
        }
      } else {
        defer = true;
      }
    } else {
      defer = true;
    }
    if (defer && tid == 0) {
      const unsigned long long at = atomicAdd(&a.ctr[1], 1ull);
      a.def_key[at] = i;
      a.def_c[at] = c;
      a.found[i] = 0;
      a.cnt[i] = 0;
      a.ptr[i] = 0;
    }
  }
}

// The sources of deferred key h again, written to src_ptr / src_len from src_off[h] on, and its
// heavy-union group (gin[h], rec[h]); flags[0] = 1 if one list is 2^32 values or longer.
__global__ void __launch_bounds__(256)
k8_sources_kernel(const K8Args a, uint32_t ndef, const uint64_t* __restrict__ src_off,
                  uint64_t* __restrict__ src_ptr, uint32_t* __restrict__ src_len,
                  GroupIn* __restrict__ gin, uint32_t* __restrict__ rec, uint32_t* flags) {
  __shared__ uint64_t s_ws[256 / 32 + 2];
  __shared__ uint32_t s_ws32[256 / 32 + 2];
  for (uint32_t h = blockIdx.x; h < ndef; h += gridDim.x) {
    const uint32_t i = a.def_key[h];
    const uint32_t k0 = a.koff[i], kn = a.koff[i + 1] - k0;
    const uint64_t off = src_off[h];
    uint64_t L;
    const uint32_t c = find_sources(a.segs, a.k, a.kb + k0, kn, L, s_ws, s_ws32,
                                    [&](uint32_t j, uint64_t p, uint64_t len, uint64_t) {
                                      if (len > 0xFFFFFFFFull) atomicExch(&flags[0], 1u);
                                      src_ptr[off + j] = p;
                                      src_len[off + j] = (uint32_t)len;
                                    });
    if (threadIdx.x == 0) {
      GroupIn g;
      g.inst = 0;
      g.tlen = 0;
      g.src = (uint32_t)off;
      g.c = c;
      g.L = 0xFFFFFFFFu;
      g.pst = 0;
      g.eslot = 0;
      g.pad = 0;
      gin[h] = g;
      rec[h] = h;
    }
  }
}

__global__ void __launch_bounds__(256)
k8_deferred_done(const K8Args a, uint32_t ndef, const GroupRec* __restrict__ recs) {
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= ndef) return;
  const uint32_t i = a.def_key[h];
  const GroupRec r = recs[h];
  a.found[i] = (r.cnt || a.keep_empty) ? 1 : 0;
  a.cnt[i] = r.cnt;
  a.ptr[i] = r.dec;
}

// grid (x = CTAs per key, y = key - y0): copy key y0 + y's list to its place
__global__ void __launch_bounds__(256)
k8_place(const uint64_t* __restrict__ ptr, const uint64_t* __restrict__ off, uint32_t y0,
         uint32_t* __restrict__ out) {
  const uint32_t i = y0 + blockIdx.y;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(ptr[i]);
  const uint64_t n = off[i + 1] - off[i];
  uint32_t* dst = out + off[i];
  for (uint64_t e = (uint64_t)blockIdx.x * 256 + threadIdx.x; e < n; e += (uint64_t)gridDim.x * 256)
    dst[e] = src[e];
}

int lookup_ctas() {
  static int per_sm = 0;
  if (!per_sm) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k8_lookup_kernel, 256, 0) != cudaSuccess || n < 1)
      n = 1;
    per_sm = n;
  }
  return per_sm * kNumSMs;
}

}  // namespace

int k8_lookup(const SegDesc* d_segs, int k, uint64_t n_post, const uint8_t* d_kb,
              const uint32_t* d_koff, uint32_t nkeys, const RemovedSet& rem, bool keep_empty,
              LookupOut& out, cudaStream_t s) {
  out.total = 0;
  out.postings_in = 0;
  const uint64_t pool_cap =
      std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)nkeys * kLookupCap, n_post));
  DevBuf<uint64_t> cnt, ptr, d_tot;
  DevBuf<uint32_t> pool, def_key, def_c;
  DevBuf<unsigned long long> ctr;
  II2_TRY(out.found.alloc_scratch(nkeys, s));
  II2_TRY(out.post_off.alloc_scratch((size_t)nkeys + 1, s));
  II2_TRY(cnt.alloc_scratch((size_t)nkeys + 1, s));
  II2_TRY(ptr.alloc_scratch(nkeys, s));
  II2_TRY(pool.alloc_scratch(pool_cap, s));
  II2_TRY(def_key.alloc_scratch(nkeys, s));
  II2_TRY(def_c.alloc_scratch(nkeys, s));
  II2_TRY(ctr.alloc_scratch(4, s));
  II2_TRY(d_tot.alloc_scratch(1, s));
  II2_CUDA_TRY(cudaMemsetAsync(ctr.p, 0, 4 * 8, s));
  II2_CUDA_TRY(cudaMemsetAsync(cnt.p + nkeys, 0, 8, s));
  K8Args a;
  a.segs = d_segs;
  a.k = k;
  a.kb = d_kb;
  a.koff = d_koff;
  a.nkeys = nkeys;
  a.rem = rem;
  a.keep_empty = keep_empty ? 1 : 0;
  a.found = out.found.p;
  a.cnt = cnt.p;
  a.ptr = ptr.p;
  a.pool = pool.p;
  a.pool_cap = pool_cap;
  a.ctr = ctr.p;
  a.def_key = def_key.p;
  a.def_c = def_c.p;
  {
    ProfScope scope("k8_lookup", s);
    k8_lookup_kernel<<<(unsigned)std::min<uint64_t>(nkeys, (uint64_t)lookup_ctas()), 256, 0, s>>>(a);
    II2_LAUNCHED();
  }
  // counts -> offsets (the deferred keys' counts are still 0: without any, these are final)
  auto offsets = [&]() -> int {
    II2_CUDA_TRY(cudaMemcpyAsync(out.post_off.p, cnt.p, ((size_t)nkeys + 1) * 8,
                                 cudaMemcpyDeviceToDevice, s));
    return exclusive_scan_u64(out.post_off.p, (uint64_t)nkeys + 1, d_tot.p, s);
  };
  II2_TRY(offsets());
  uint64_t* const h = pinned_scratch();
  if (!h) return II2_ERR_NOMEM;
  II2_TRY(small_copy(h, ctr.p, 24, s));
  II2_TRY(small_copy(h + 3, d_tot.p, 8, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  const uint32_t ndef = (uint32_t)h[1];
  out.postings_in = h[2];
  out.total = h[3];
  DevBuf<uint32_t> large_tmp, large_enc;  // the heavy unions (until they are placed)
  if (ndef) {
    ProfScope scope("k8_deferred", s);
    // their source counts size the source arrays of the heavy union
    std::vector<uint32_t> h_c(ndef);
    std::vector<uint64_t> h_off(ndef);
    II2_CUDA_TRY(cudaMemcpyAsync(h_c.data(), def_c.p, (size_t)ndef * 4, cudaMemcpyDeviceToHost, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    uint64_t nsrc = 0;
    for (uint32_t i = 0; i < ndef; i++) {
      h_off[i] = nsrc;
      nsrc += h_c[i];
    }
    if (nsrc >= (1ull << 32)) {
      set_last_error("lookup: %llu (key, segment) sources of heavy keys (max 2^32-1)",
                     (unsigned long long)nsrc);
      return II2_ERR_UNSUPPORTED;
    }
    DevBuf<uint64_t> src_off, src_ptr;
    DevBuf<uint32_t> src_len, rec, flags;
    DevBuf<GroupIn> gin;
    DevBuf<GroupRec> recs;
    II2_TRY(src_off.alloc_scratch(ndef, s));
    II2_TRY(src_ptr.alloc_scratch(nsrc, s));
    II2_TRY(src_len.alloc_scratch(nsrc, s));
    II2_TRY(rec.alloc_scratch(ndef, s));
    II2_TRY(flags.alloc_scratch(2, s));
    II2_TRY(gin.alloc_scratch(ndef, s));
    II2_TRY(recs.alloc_scratch(ndef, s));
    II2_CUDA_TRY(cudaMemcpyAsync(src_off.p, h_off.data(), (size_t)ndef * 8, cudaMemcpyHostToDevice, s));
    II2_CUDA_TRY(cudaMemsetAsync(flags.p, 0, 8, s));
    k8_sources_kernel<<<(unsigned)std::min<uint64_t>(ndef, (uint64_t)lookup_ctas()), 256, 0, s>>>(
        a, ndef, src_off.p, src_ptr.p, src_len.p, gin.p, rec.p, flags.p);
    II2_LAUNCHED();
    uint32_t* const h_flag = reinterpret_cast<uint32_t*>(h + 4);
    h_flag[0] = 0;
    II2_TRY(small_copy(h_flag, flags.p, 8, s));
    LargeArgs la;
    la.rec = rec.p;
    la.bucket = nullptr;
    la.gin = gin.p;
    la.src_ptr = src_ptr.p;
    la.src_len = src_len.p;
    la.recs = recs.p;
    la.rem = rem;
    la.want_enc = 0;
    la.keep_empty = keep_empty ? 1 : 0;
    la.always_sort = 0;  // a single source passes through as stored (survey Q4)
    la.presorted = nullptr;
    la.bk_raw = nullptr;
    la.nb1 = 0;
    II2_TRY(k2_large_run(la, ndef, large_tmp, large_enc, s));  // (synchronises)
    if (h_flag[0]) {
      set_last_error("lookup: one segment holds 2^32 or more postings under a key");
      return II2_ERR_UNSUPPORTED;
    }
    k8_deferred_done<<<div_up(ndef, 256), 256, 0, s>>>(a, ndef, recs.p);
    II2_LAUNCHED();
    II2_TRY(offsets());
    II2_TRY(small_copy(h + 3, d_tot.p, 8, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    out.total = h[3];
  }
  II2_TRY(out.post.alloc_scratch(out.total, s));
  if (out.total) {
    ProfScope scope("k8_place", s);
    const unsigned gx = (unsigned)std::max<uint64_t>(
        1, std::min<uint64_t>(1024, (out.total / nkeys + 2047) / 2048));
    for (uint32_t y0 = 0; y0 < nkeys; y0 += 32768) {
      const uint32_t ny = std::min<uint32_t>(32768, nkeys - y0);
      k8_place<<<dim3(gx, ny), 256, 0, s>>>(ptr.p, out.post_off.p, y0, out.post.p);
      II2_LAUNCHED();
    }
  }
  return II2_OK;
}

}  // namespace ii2
