// k7_ingest.cu — K7: a batch of ingested documents becomes direct-mode segments on the device.
//
// Replaces, for D documents at once, the per-document work of Shard.Put (shard.go:33-67):
// slices.SortFunc(terms, bytes.Compare) (:34) and one direct-mode segment per document whose
// every term carries the document's value (file/writer.go:34-40).  The reference writes D FST
// files and folds them later in Shard.Merge; here the D sorted dictionaries are built in HBM
// (one segmented sort over all documents) and handed straight to the merge pipeline, so
// "Put x D + Merge" is one call (ii2_ingest, SURVEY 8f row 4).
//
// Sort: records (16-byte big-endian key window, term index), one bitonic network per document
// — 2048-record tiles in shared memory, direction-free global stages beyond a tile (the same
// network as the heavy-term union of k12_union.cu) — ordered by bytes.Compare: key window, then
// the bytes past it, then length.  A term repeated inside one document is kept once: vellum
// collapses a repeated Insert of the same key with the same output into the one existing path
// (the reference's own count of such a segment is off by one; reads see the term once).
// Integer/byte work, HBM-bound.
#include <algorithm>
#include <vector>

#include "ingest.cuh"
#include "keys.cuh"

namespace ii2 {

namespace {

constexpr uint32_t K7_TILE = 2048;
constexpr int K7_THREADS = 512;

struct K7Args {
  const uint8_t* tb;     // all documents' term bytes (as given, unsorted)
  const uint32_t* toff;  // [N + 1] global byte offsets
  const uint64_t* doff;  // [D + 1] first term of every document
  uint64_t* hi;          // [N] sort records
  uint64_t* lo;
  uint32_t* idx;
  uint64_t n;
  int d;
};

// bytes.Compare of the terms behind two records
__device__ __forceinline__ int k7_cmp(const K7Args& a, uint64_t ha, uint64_t la, uint32_t ia,
                                      uint64_t hb, uint64_t lb, uint32_t ib) {
  if (ha != hb) return ha < hb ? -1 : 1;
  if (la != lb) return la < lb ? -1 : 1;
  const uint32_t oa = a.toff[ia], na = a.toff[ia + 1] - oa;
  const uint32_t ob = a.toff[ib], nb = a.toff[ib + 1] - ob;
  if (na > 16 && nb > 16) return term_compare(a.tb + oa + 16, na - 16, a.tb + ob + 16, nb - 16);
  return na < nb ? -1 : (na > nb ? 1 : 0);
}

__global__ void __launch_bounds__(256) k7_keys(const K7Args a) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= a.n) return;
  const uint32_t o = a.toff[i], len = a.toff[i + 1] - o;
  uint64_t h, l;
  load_key16(a.tb, o, len, 0, h, l);
  a.hi[i] = h;
  a.lo[i] = l;
  a.idx[i] = (uint32_t)i;
}

// grid (x = tiles, y = document): sort every aligned tile of the document in shared memory
__global__ void __launch_bounds__(K7_THREADS) k7_tile_sort(const K7Args a) {
  __shared__ uint64_t s_hi[K7_TILE], s_lo[K7_TILE];
  __shared__ uint32_t s_idx[K7_TILE];
  __shared__ uint16_t perm[K7_TILE];
  const uint64_t d0 = a.doff[blockIdx.y], n = a.doff[blockIdx.y + 1] - d0;
  for (uint64_t t0 = (uint64_t)blockIdx.x * K7_TILE; t0 < n; t0 += (uint64_t)gridDim.x * K7_TILE) {
    const uint32_t m = (uint32_t)((n - t0) < K7_TILE ? (n - t0) : K7_TILE);
    for (uint32_t i = threadIdx.x; i < m; i += K7_THREADS) {
      s_hi[i] = a.hi[d0 + t0 + i];
      s_lo[i] = a.lo[d0 + t0 + i];
      s_idx[i] = a.idx[d0 + t0 + i];
      perm[i] = (uint16_t)i;
    }
    __syncthreads();
    bitonic_sort_any(perm, m, threadIdx.x, (uint32_t)K7_THREADS,
                     [&](uint16_t x, uint16_t y) {
                       return k7_cmp(a, s_hi[x], s_lo[x], s_idx[x], s_hi[y], s_lo[y], s_idx[y]) < 0;
                     },
                     [] { __syncthreads(); });
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < m; i += K7_THREADS) {
      const uint32_t p = perm[i];
      a.hi[d0 + t0 + i] = s_hi[p];
      a.lo[d0 + t0 + i] = s_lo[p];
      a.idx[d0 + t0 + i] = s_idx[p];
    }
    __syncthreads();
  }
}

// one global stage of the direction-free network: flip (kk, j == 0) or half-cleaner j
__global__ void __launch_bounds__(256) k7_stage(const K7Args a, uint64_t kk, uint64_t j) {
  const uint64_t d0 = a.doff[blockIdx.y], n = a.doff[blockIdx.y + 1] - d0;
  if ((kk >> 1) >= n) return;
  const uint64_t half = j ? j : (kk >> 1);
  const uint64_t limit = (n + 1) / 2 + half;
  for (uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x; t < limit; t += (uint64_t)gridDim.x * 256) {
    uint64_t i, l;
    if (j == 0) {
      i = (t / half) * kk + (t % half);
      l = i ^ (kk - 1);
    } else {
      i = (t / j) * (j << 1) + (t % j);
      l = i + j;
    }
    if (l < n && i < n) {
      const uint64_t hx = a.hi[d0 + i], lx = a.lo[d0 + i], hy = a.hi[d0 + l], ly = a.lo[d0 + l];
      const uint32_t ix = a.idx[d0 + i], iy = a.idx[d0 + l];
      if (k7_cmp(a, hy, ly, iy, hx, lx, ix) < 0) {
        a.hi[d0 + i] = hy;
        a.lo[d0 + i] = ly;
        a.idx[d0 + i] = iy;
        a.hi[d0 + l] = hx;
        a.lo[d0 + l] = lx;
        a.idx[d0 + l] = ix;
      }
    }
  }
}

// finish block size kk inside shared memory: half-cleaners j = K7_TILE/2 .. 1
__global__ void __launch_bounds__(K7_THREADS) k7_tile_merge(const K7Args a, uint64_t kk) {
  __shared__ uint64_t s_hi[K7_TILE], s_lo[K7_TILE];
  __shared__ uint32_t s_idx[K7_TILE];
  const uint64_t d0 = a.doff[blockIdx.y], n = a.doff[blockIdx.y + 1] - d0;
  if ((kk >> 1) >= n) return;
  for (uint64_t t0 = (uint64_t)blockIdx.x * K7_TILE; t0 < n; t0 += (uint64_t)gridDim.x * K7_TILE) {
    const uint32_t m = (uint32_t)((n - t0) < K7_TILE ? (n - t0) : K7_TILE);
    for (uint32_t i = threadIdx.x; i < m; i += K7_THREADS) {
      s_hi[i] = a.hi[d0 + t0 + i];
      s_lo[i] = a.lo[d0 + t0 + i];
      s_idx[i] = a.idx[d0 + t0 + i];
    }
    __syncthreads();
    for (uint32_t j = K7_TILE / 2; j >= 1; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < K7_TILE / 2; t += K7_THREADS) {
        const uint32_t i = (t / j) * (j << 1) + (t % j);
        const uint32_t l = i + j;
        if (l < m) {
          if (k7_cmp(a, s_hi[l], s_lo[l], s_idx[l], s_hi[i], s_lo[i], s_idx[i]) < 0) {
            const uint64_t h = s_hi[i], w = s_lo[i];
            const uint32_t x = s_idx[i];
            s_hi[i] = s_hi[l];
            s_lo[i] = s_lo[l];
            s_idx[i] = s_idx[l];
            s_hi[l] = h;
            s_lo[l] = w;
            s_idx[l] = x;
          }
        }
      }
      __syncthreads();
    }
    for (uint32_t i = threadIdx.x; i < m; i += K7_THREADS) {
      a.hi[d0 + t0 + i] = s_hi[i];
      a.lo[d0 + t0 + i] = s_lo[i];
      a.idx[d0 + t0 + i] = s_idx[i];
    }
    __syncthreads();
  }
}

__device__ __forceinline__ int k7_doc_of(const uint64_t* __restrict__ doff, int d, uint64_t p) {
  int lo = 0, hi = d;  // last document with doff <= p (empty documents share their start)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (doff[mid + 1] <= p)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// keep[p] = 1 for the first record of every distinct term of a document; klen[p] = its bytes
__global__ void __launch_bounds__(256)
k7_mark(const K7Args a, uint64_t* __restrict__ keep, uint64_t* __restrict__ klen) {
  const uint64_t p = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (p > a.n) return;
  if (p == a.n) {
    keep[p] = klen[p] = 0;
    return;
  }
  const int d = k7_doc_of(a.doff, a.d, p);
  bool first = p == a.doff[d];
  if (!first)
    first = k7_cmp(a, a.hi[p - 1], a.lo[p - 1], a.idx[p - 1], a.hi[p], a.lo[p], a.idx[p]) != 0;
  const uint32_t i = a.idx[p];
  keep[p] = first ? 1u : 0u;
  klen[p] = first ? a.toff[i + 1] - a.toff[i] : 0u;
}

struct K7Emit {
  const uint64_t* pos;   // [N + 1] exclusive scan of keep
  const uint64_t* boff;  // [N + 1] exclusive scan of klen
  const uint32_t* vals;  // [D]
  uint8_t* o_tb;
  uint32_t* o_toff;
  uint32_t* o_post;
  uint64_t* o_poff;
  uint64_t* o_first;     // [D + 1] first kept term of every document
};

// one warp per sorted record: place the kept ones
__global__ void __launch_bounds__(256) k7_emit(const K7Args a, const K7Emit e) {
  const uint64_t p = ((uint64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  const unsigned lane = lane_id();
  if (p > a.n) return;
  const uint64_t r = e.pos[p];
  if (p == a.n) {
    if (lane == 0) {
      e.o_toff[r] = (uint32_t)e.boff[p];
      e.o_poff[r] = r;
      e.o_first[a.d] = r;
      for (int q = a.d - 1; q >= 0 && a.doff[q] == p; q--) e.o_first[q] = r;  // empty tail
    }
    return;
  }
  const int d = k7_doc_of(a.doff, a.d, p);
  if (lane == 0 && p == a.doff[d]) {
    // documents that start here: d and the empty ones before it that share this position
    e.o_first[d] = r;
    for (int q = d - 1; q >= 0 && a.doff[q] == p; q--) e.o_first[q] = r;
  }
  if (e.pos[p + 1] == r) return;  // repeated term
  const uint32_t i = a.idx[p];
  const uint32_t o = a.toff[i], len = a.toff[i + 1] - o;
  const uint32_t dst = (uint32_t)e.boff[p];
  for (uint32_t q = lane; q < len; q += 32) e.o_tb[dst + q] = a.tb[o + q];
  if (lane == 0) {
    e.o_toff[r] = dst;
    e.o_post[r] = e.vals[d];
    e.o_poff[r] = r;
  }
}

// sort every document's records by bytes.Compare of their terms: a.hi / a.lo / a.idx hold the
// sorted records afterwards (maxL = the longest document)
int k7_sort(const K7Args& a, uint64_t maxL, cudaStream_t s) {
  if (!a.n) return II2_OK;
  ProfScope scope("k7_sort", s);
  k7_keys<<<div_up(a.n, 256), 256, 0, s>>>(a);
  II2_LAUNCHED();
  for (int y0 = 0; y0 < a.d; y0 += 32768) {  // grid.y limit
    const int ny = std::min(32768, a.d - y0);
    K7Args b = a;
    b.doff += y0;
    const unsigned gx = (unsigned)std::max<uint64_t>(
        1, std::min<uint64_t>((maxL + K7_TILE - 1) / K7_TILE, 2048));
    const dim3 grid(gx, ny);
    k7_tile_sort<<<grid, K7_THREADS, 0, s>>>(b);
    II2_LAUNCHED();
    for (uint64_t kk = 2ull * K7_TILE; (kk >> 1) < maxL; kk <<= 1) {
      k7_stage<<<grid, 256, 0, s>>>(b, kk, 0);
      II2_LAUNCHED();
      for (uint64_t j = kk >> 2; j >= K7_TILE; j >>= 1) {
        k7_stage<<<grid, 256, 0, s>>>(b, kk, j);
        II2_LAUNCHED();
      }
      k7_tile_merge<<<grid, K7_THREADS, 0, s>>>(b, kk);
      II2_LAUNCHED();
    }
  }
  return II2_OK;
}

}  // namespace

int k7_ingest_sort(const uint8_t* d_tb, const uint32_t* d_toff, const uint64_t* d_doff,
                   const uint64_t* h_doff, const uint32_t* d_vals, int D, uint64_t N, uint64_t TB,
                   IngestOut& out, cudaStream_t s) {
  out.first.assign((size_t)D + 1, 0);
  II2_TRY(out.tb.alloc((size_t)TB, s, 32));
  II2_TRY(out.toff.alloc((size_t)N + 1, s));
  II2_TRY(out.post.alloc((size_t)N, s, 16));
  II2_TRY(out.poff.alloc((size_t)N + 1, s));
  DevBuf<uint64_t> hi, lo, keep, klen, d_first;
  DevBuf<uint32_t> idx;
  II2_TRY(hi.alloc_scratch((size_t)N, s));
  II2_TRY(lo.alloc_scratch((size_t)N, s));
  II2_TRY(idx.alloc_scratch((size_t)N, s));
  II2_TRY(keep.alloc_scratch((size_t)N + 1, s));
  II2_TRY(klen.alloc_scratch((size_t)N + 1, s));
  II2_TRY(d_first.alloc_scratch((size_t)D + 1, s));
  K7Args a;
  a.tb = d_tb;
  a.toff = d_toff;
  a.doff = d_doff;
  a.hi = hi.p;
  a.lo = lo.p;
  a.idx = idx.p;
  a.n = N;
  a.d = D;
  uint64_t maxL = 0;
  for (int d = 0; d < D; d++) maxL = std::max(maxL, h_doff[d + 1] - h_doff[d]);
  II2_TRY(k7_sort(a, maxL, s));
  ProfScope scope("k7_build", s);
  k7_mark<<<div_up(N + 1, 256), 256, 0, s>>>(a, keep.p, klen.p);
  II2_LAUNCHED();
  DevBuf<uint64_t> d_tot;
  II2_TRY(d_tot.alloc_scratch(2, s));
  II2_TRY(exclusive_scan_u64(keep.p, N + 1, d_tot.p, s));
  II2_TRY(exclusive_scan_u64(klen.p, N + 1, d_tot.p + 1, s));
  K7Emit e;
  e.pos = keep.p;
  e.boff = klen.p;
  e.vals = d_vals;
  e.o_tb = out.tb.p;
  e.o_toff = out.toff.p;
  e.o_post = out.post.p;
  e.o_poff = out.poff.p;
  e.o_first = d_first.p;
  k7_emit<<<div_up((N + 1) * 32, 256), 256, 0, s>>>(a, e);
  II2_LAUNCHED();
  II2_CUDA_TRY(cudaMemcpyAsync(out.first.data(), d_first.p, ((size_t)D + 1) * 8,
                               cudaMemcpyDeviceToHost, s));
  uint64_t h_tot[2] = {0, 0};
  II2_CUDA_TRY(cudaMemcpyAsync(h_tot, d_tot.p, 16, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  out.n_terms = h_tot[0];
  out.n_bytes = h_tot[1];
  return II2_OK;
}

int k7_sort_distinct(const uint8_t* d_tb, const uint32_t* d_toff, const uint64_t* d_doff, int D,
                     uint64_t N, uint64_t maxL, uint32_t* idx, uint64_t* keep, uint64_t* klen,
                     cudaStream_t s) {
  DevBuf<uint64_t> hi, lo;
  II2_TRY(hi.alloc_scratch((size_t)N, s));
  II2_TRY(lo.alloc_scratch((size_t)N, s));
  K7Args a;
  a.tb = d_tb;
  a.toff = d_toff;
  a.doff = d_doff;
  a.hi = hi.p;
  a.lo = lo.p;
  a.idx = idx;
  a.n = N;
  a.d = D;
  II2_TRY(k7_sort(a, maxL, s));
  k7_mark<<<div_up(N + 1, 256), 256, 0, s>>>(a, keep, klen);
  II2_LAUNCHED();
  return II2_OK;
}

}  // namespace ii2
