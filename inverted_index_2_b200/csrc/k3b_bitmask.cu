// k3b_bitmask.cu — K3b: file/bitmask.go Bitmask[uint32] on the device.
//
//   Put  (file/bitmask.go:53-59)  idx = first dictionary position of every value, appended on
//        miss in input order (:64-71); roaring bitmap of the indexes; portable serialisation.
//   Get  (file/bitmask.go:30-49)  parse ONE serialised bitmap from the front of the buffer,
//        ascending indexes -> dictionary values; "bitmask is out of bound" (:41-44).
//
// How the sequential reference maps onto the GPU without changing a byte of the result:
//   - slices.Index (O(dictionary) per value) becomes a device hash table value -> FIRST index
//     (64-bit slots value<<32|index, atomicMin keeps the smallest index, so duplicate
//     dictionary entries and duplicate input values resolve like the linear scan).
//   - append-on-miss in input order = stable compaction: every missing value is inserted with
//     the provisional index D+i, the smallest i per distinct value wins, an exclusive scan over
//     the winners gives the final dictionary slot.
//   - roaring's container state after a sequence of Add() calls depends only on the final set
//     (RoaringBitmap/roaring v1.9.4: array while cardinality <= 4096, bitmap above, a full
//     bitmap container becomes the run [0,65535]; RunOptimize is never called), so the indexes
//     are OR-ed into a plain bit set and each 65536-bit chunk is serialised by its popcount.
// Integer/byte work, HBM-bound: per Put 4 B/value in, hash probes in L2, bit set + output.
#include <algorithm>
#include <memory>

#include "runtime.cuh"

using namespace ii2;

struct ii2_bitmask {
  int device = ctx_current_device();  // where its arrays live: every operation runs there
  uint64_t n = 0;  // dictionary length
  DevBuf<uint32_t> values;
  uint64_t values_cap = 0;
  DevBuf<unsigned long long> table;
  uint64_t table_cap = 0;  // slots, power of two
  // Direct-address inverse of the dictionary, inv[v] = FIRST index of value v (0xFFFFFFFF: not
  // in the dictionary), kept while the largest value is at most a few times the dictionary
  // length (a universe of document ids, file/bitmask_test.go:15-21): a Put whose values are all
  // in the dictionary is then ONE probe per value instead of four passes of hash probes.
  DevBuf<uint32_t> inv;
  uint64_t inv_len = 0;    // maxv + 1, 0 = no inverse
  uint64_t inv_for_n = 0;  // dictionary length the inverse was built for
};

namespace {

constexpr unsigned long long BM_EMPTY = ~0ull;
constexpr uint32_t BM_NOT_FOUND = 0xFFFFFFFFu;
constexpr int BM_THREADS = 256;
constexpr uint32_t CHUNK_WORDS = 2048;  // 65536 bits as u32 words

__device__ __forceinline__ uint64_t bm_hash(uint32_t x) {
  uint64_t h = (uint64_t)x * 0x9E3779B97F4A7C15ull;
  return h ^ (h >> 29);
}

__device__ __forceinline__ void tbl_insert_min(unsigned long long* t, uint64_t mask, uint32_t v,
                                               uint32_t idx) {
  const unsigned long long ent = ((unsigned long long)v << 32) | idx;
  uint64_t h = bm_hash(v) & mask;
  for (;;) {
    unsigned long long e = *reinterpret_cast<volatile unsigned long long*>(t + h);
    if (e == BM_EMPTY) {
      e = atomicCAS(t + h, BM_EMPTY, ent);
      if (e == BM_EMPTY) return;
    }
    if ((uint32_t)(e >> 32) == v) {
      atomicMin(t + h, ent);
      return;
    }
    h = (h + 1) & mask;
  }
}

// slot of value v (must be present)
__device__ __forceinline__ uint64_t tbl_slot(const unsigned long long* t, uint64_t mask, uint32_t v) {
  uint64_t h = bm_hash(v) & mask;
  for (;;) {
    unsigned long long e = t[h];
    if (e == BM_EMPTY || (uint32_t)(e >> 32) == v) return h;
    h = (h + 1) & mask;
  }
}

__device__ __forceinline__ uint32_t tbl_find(const unsigned long long* t, uint64_t mask, uint32_t v) {
  unsigned long long e = t[tbl_slot(t, mask, v)];
  return e == BM_EMPTY ? BM_NOT_FOUND : (uint32_t)e;
}

__global__ void __launch_bounds__(BM_THREADS)
k_bm_build(unsigned long long* t, uint64_t mask, const uint32_t* __restrict__ values, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) tbl_insert_min(t, mask, values[i], (uint32_t)i);
}

// provisional insert: value i -> D + i
__global__ void __launch_bounds__(BM_THREADS)
k_bm_put_insert(unsigned long long* t, uint64_t mask, const uint32_t* __restrict__ vals, uint64_t n,
                uint32_t D) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) tbl_insert_min(t, mask, vals[i], D + (uint32_t)i);
}

// winner[i] = 1 iff input position i is the first occurrence of a value missing from the
// dictionary (the position whose append slices.Index would have caused, bitmask.go:66-69)
__global__ void __launch_bounds__(BM_THREADS)
k_bm_put_flag(const unsigned long long* __restrict__ t, uint64_t mask,
              const uint32_t* __restrict__ vals, uint64_t n, uint32_t D, uint64_t* __restrict__ win) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  win[i] = (i < n && tbl_find(t, mask, vals[i]) == D + (uint32_t)i) ? 1u : 0u;
}

// final index of every value; winners append to the dictionary; bit set
__global__ void __launch_bounds__(BM_THREADS)
k_bm_put_resolve(const unsigned long long* __restrict__ t, uint64_t mask,
                 const uint32_t* __restrict__ vals, uint64_t n, uint32_t D,
                 const uint64_t* __restrict__ rank, uint32_t* __restrict__ values,
                 uint32_t* __restrict__ bits) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = vals[i];
  uint32_t e = tbl_find(t, mask, v);
  if (e >= D) {
    const uint32_t w = e - D;
    e = D + (uint32_t)rank[w];
    if (w == (uint32_t)i) values[e] = v;
  }
  atomicOr(&bits[e >> 5], 1u << (e & 31u));
}

// provisional -> final index in the table (after every lookup of the resolve pass)
__global__ void __launch_bounds__(BM_THREADS)
k_bm_put_fixup(unsigned long long* t, uint64_t mask, const uint32_t* __restrict__ vals, uint64_t n,
               uint32_t D, const uint64_t* __restrict__ rank) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = vals[i];
  const uint64_t h = tbl_slot(t, mask, v);
  if ((uint32_t)t[h] == D + (uint32_t)i)
    t[h] = ((unsigned long long)v << 32) | (D + (uint32_t)rank[i]);
}

// ---- direct-address inverse -------------------------------------------------------------------
__global__ void __launch_bounds__(BM_THREADS)
k_bm_max(const uint32_t* __restrict__ values, uint64_t n, uint32_t* __restrict__ out) {
  uint32_t m = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (uint64_t)gridDim.x * blockDim.x)
    m = max(m, values[i]);
  m = __reduce_max_sync(0xffffffffu, m);
  if (lane_id() == 0 && m) atomicMax(out, m);
}
__global__ void __launch_bounds__(BM_THREADS)
k_bm_inv_build(const uint32_t* __restrict__ values, uint64_t n, uint32_t* __restrict__ inv) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicMin(&inv[values[i]], (uint32_t)i);  // slices.Index: the first occurrence
}
// one probe per value; miss[0] counts values that are not in the dictionary (the caller then
// takes the general path, which appends them in input order)
__global__ void __launch_bounds__(BM_THREADS)
k_bm_put_direct(const uint32_t* __restrict__ inv, uint64_t inv_len, const uint32_t* __restrict__ vals,
                uint64_t n, uint32_t* __restrict__ bits, uint32_t* __restrict__ miss) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = vals[i];
  const uint32_t e = v < inv_len ? __ldg(inv + v) : BM_NOT_FOUND;
  if (e == BM_NOT_FOUND)
    atomicAdd(miss, 1u);
  else
    atomicOr(&bits[e >> 5], 1u << (e & 31u));
}

// cardinality of every 65536-bit chunk
__global__ void __launch_bounds__(BM_THREADS)
k_bm_chunk_card(const uint32_t* __restrict__ bits, uint32_t* __restrict__ card) {
  __shared__ uint32_t ws[BM_THREADS / 32 + 2];
  const uint32_t* w = bits + (uint64_t)blockIdx.x * CHUNK_WORDS;
  uint32_t c = 0;
  for (uint32_t i = threadIdx.x; i < CHUNK_WORDS; i += BM_THREADS) c += __popc(w[i]);
  uint32_t tot;
  block_exclusive_scan(c, ws, tot);
  if (threadIdx.x == 0) card[blockIdx.x] = tot;
}

__device__ __forceinline__ uint32_t payload_bytes(uint32_t card) {
  // getSizeInBytesFromCardinality / run container [0,65535] = n_runs + one (start, length-1)
  return card == 0 ? 0u : card <= 4096u ? 2u * card : card < 65536u ? 8192u : 6u;
}

// One CTA over all chunks: container index + payload offset per non-empty chunk.
// totals: [0] containers [1] payload bytes [2] has_run
__global__ void __launch_bounds__(1024)
k_bm_chunk_scan(const uint32_t* __restrict__ card, uint32_t nchunks, uint32_t* __restrict__ cidx,
                uint64_t* __restrict__ poff, uint32_t* __restrict__ cont_chunk,
                uint64_t* __restrict__ totals) {
  __shared__ uint64_t ws[1024 / 32 + 2];
  __shared__ uint32_t s_run;
  if (threadIdx.x == 0) s_run = 0;
  __syncthreads();
  uint64_t run_c = 0, run_p = 0;
  for (uint32_t base = 0; base < nchunks; base += 1024) {
    const uint32_t ch = base + threadIdx.x;
    const uint32_t c = ch < nchunks ? card[ch] : 0u;
    if (c == 65536u) s_run = 1;
    uint64_t tot_c, tot_p;
    const uint64_t ex_c = block_exclusive_scan<uint64_t>(c ? 1u : 0u, ws, tot_c);
    const uint64_t ex_p = block_exclusive_scan<uint64_t>(payload_bytes(c), ws, tot_p);
    if (c) {
      cidx[ch] = (uint32_t)(run_c + ex_c);
      poff[ch] = run_p + ex_p;
      cont_chunk[run_c + ex_c] = ch;
    }
    run_c += tot_c;
    run_p += tot_p;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    totals[0] = run_c;
    totals[1] = run_p;
    totals[2] = s_run;
  }
}

// little-endian stores at any byte alignment (the run-cookie header can be odd-sized)
__device__ __forceinline__ void st16(uint8_t* p, uint32_t v) {
  if (reinterpret_cast<uintptr_t>(p) & 1u) {
    p[0] = (uint8_t)v;
    p[1] = (uint8_t)(v >> 8);
  } else {
    *reinterpret_cast<uint16_t*>(p) = (uint16_t)v;
  }
}
__device__ __forceinline__ void st32(uint8_t* p, uint32_t v) {
  st16(p, v & 0xFFFFu);
  st16(p + 2, v >> 16);
}
__device__ __forceinline__ uint32_t ld16(const uint8_t* p) {
  if (reinterpret_cast<uintptr_t>(p) & 1u) return (uint32_t)p[0] | ((uint32_t)p[1] << 8);
  return *reinterpret_cast<const uint16_t*>(p);
}
__device__ __forceinline__ uint32_t ld32(const uint8_t* p) { return ld16(p) | (ld16(p + 2) << 16); }

// roaringArray.writeTo header: cookie, (run flags), descriptive header, (offset header)
__global__ void __launch_bounds__(BM_THREADS)
k_bm_header(const uint32_t* __restrict__ card, const uint64_t* __restrict__ poff,
            const uint32_t* __restrict__ cont_chunk, uint32_t nc, int has_run, uint8_t* out,
            uint32_t desc_at, uint32_t offs_at, int has_off, uint32_t data_at) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0) {
    if (has_run) {
      st16(out, 12347u);
      st16(out + 2, nc - 1);
    } else {
      st32(out, 12346u);
      st32(out + 4, nc);
    }
  }
  if (c >= nc) return;
  const uint32_t ch = cont_chunk[c];
  const uint32_t cd = card[ch];
  st16(out + desc_at + 4 * c, ch);
  st16(out + desc_at + 4 * c + 2, cd - 1);
  if (has_off) st32(out + offs_at + 4 * c, data_at + (uint32_t)poff[ch]);
  if (has_run && (c & 7u) == 0) {
    uint32_t f = 0;
    for (uint32_t j = 0; j < 8 && c + j < nc; j++)
      if (card[cont_chunk[c + j]] == 65536u) f |= 1u << j;
    out[4 + (c >> 3)] = (uint8_t)f;
  }
}

// payloads: one CTA per container
__global__ void __launch_bounds__(BM_THREADS)
k_bm_payload(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ card,
             const uint64_t* __restrict__ poff, const uint32_t* __restrict__ cont_chunk,
             uint8_t* out, uint32_t data_at) {
  __shared__ uint32_t ws[BM_THREADS / 32 + 2];
  const uint32_t ch = cont_chunk[blockIdx.x];
  const uint32_t cd = card[ch];
  const uint32_t* w = bits + (uint64_t)ch * CHUNK_WORDS;
  uint8_t* dst = out + data_at + poff[ch];
  if (cd == 65536u) {  // run container: one run [0,65535]
    if (threadIdx.x == 0) {
      st16(dst, 1);
      st16(dst + 2, 0);
      st16(dst + 4, 65535);
    }
  } else if (cd > 4096u) {  // bitmap container: 1024 u64, little-endian == the u32 words in order
    for (uint32_t i = threadIdx.x; i < CHUNK_WORDS; i += BM_THREADS) st32(dst + 4 * i, w[i]);
  } else {  // array container: ascending u16
    constexpr uint32_t PER = CHUNK_WORDS / BM_THREADS;  // consecutive words per thread
    uint32_t word[PER];
    uint32_t c = 0;
#pragma unroll
    for (uint32_t j = 0; j < PER; j++) {
      word[j] = w[threadIdx.x * PER + j];
      c += __popc(word[j]);
    }
    uint32_t tot;
    uint32_t at = block_exclusive_scan(c, ws, tot);
#pragma unroll
    for (uint32_t j = 0; j < PER; j++) {
      uint32_t x = word[j];
      while (x) {
        const uint32_t b = __ffs(x) - 1;
        x &= x - 1;
        st16(dst + 2 * at, (threadIdx.x * PER + j) * 32 + b);
        at++;
      }
    }
  }
}

// ------------------------------------------------------------------ Get
// meta per container: type (0 array, 1 bitmap, 2 run), card, payload offset, output offset
struct GetMeta {
  uint32_t type, card;
  uint64_t pay, out;
};
// info: [0] nc [1] total values [2] error (1 corrupt)
__global__ void __launch_bounds__(1024)
k_bm_get_parse(const uint8_t* __restrict__ enc, uint64_t nenc, GetMeta* __restrict__ meta,
               uint32_t meta_cap, uint64_t* __restrict__ info) {
  __shared__ uint64_t ws[1024 / 32 + 2];
  const uint32_t tid = threadIdx.x;
  if (tid == 0) {
    info[0] = 0;
    info[1] = 0;
    info[2] = 0;
  }
  __syncthreads();
  if (nenc < 4) {
    if (tid == 0) info[2] = 1;
    return;
  }
  const uint32_t cookie = ld32(enc);
  uint64_t p, nc;
  int has_run = 0;
  if ((cookie & 0xFFFFu) == 12347u) {
    has_run = 1;
    nc = (cookie >> 16) + 1;
    p = 4 + (nc + 7) / 8;
  } else if (cookie == 12346u) {
    if (nenc < 8) {
      if (tid == 0) info[2] = 1;
      return;
    }
    nc = ld32(enc + 4);
    p = 8;
  } else {
    if (tid == 0) info[2] = 1;
    return;
  }
  if (nc > 65536 || nc > meta_cap || p + 4 * nc > nenc) {
    if (tid == 0) info[2] = 1;
    return;
  }
  const uint8_t* desc = enc + p;
  p += 4 * nc;
  if (!has_run || nc >= 4) p += 4 * nc;  // offset header: payloads are sequential anyway
  if (p > nenc) {
    if (tid == 0) info[2] = 1;
    return;
  }
  if (has_run) {  // run payload sizes live in the payload: sequential walk
    if (tid == 0) {
      uint64_t o = 0;
      int bad = 0;
      for (uint64_t i = 0; i < nc && !bad; i++) {
        GetMeta m;
        m.card = ld16(desc + 4 * i + 2) + 1;
        const bool is_run = (enc[4 + i / 8] >> (i % 8)) & 1u;
        m.type = is_run ? 2u : (m.card > 4096u ? 1u : 0u);
        m.pay = p;
        m.out = o;
        uint64_t sz;
        if (is_run) {
          if (p + 2 > nenc) { bad = 1; break; }
          sz = 2 + 4ull * ld16(enc + p);
        } else {
          sz = m.type == 1 ? 8192u : 2ull * m.card;
        }
        if (p + sz > nenc) { bad = 1; break; }
        p += sz;
        o += m.card;
        meta[i] = m;
      }
      info[0] = nc;
      info[1] = o;
      info[2] = bad;
    }
    return;
  }
  uint64_t run_p = p, run_o = 0;
  int bad = 0;
  for (uint64_t base = 0; base < nc; base += 1024) {
    const uint64_t i = base + tid;
    GetMeta m;
    m.card = i < nc ? ld16(desc + 4 * i + 2) + 1 : 0u;
    m.type = m.card > 4096u ? 1u : 0u;
    const uint64_t sz = i < nc ? (m.type == 1 ? 8192u : 2ull * m.card) : 0u;
    uint64_t tot_p, tot_o;
    const uint64_t ex_p = block_exclusive_scan(sz, ws, tot_p);
    const uint64_t ex_o = block_exclusive_scan<uint64_t>(m.card, ws, tot_o);
    if (i < nc) {
      m.pay = run_p + ex_p;
      m.out = run_o + ex_o;
      meta[i] = m;
    }
    run_p += tot_p;
    run_o += tot_o;
    if (run_p > nenc) bad = 1;
  }
  if (tid == 0) {
    info[0] = nc;
    info[1] = run_o;
    info[2] = bad;
  }
}

// one CTA per container: indexes -> dictionary values.  err: 1 corrupt, 2 out of bound
__global__ void __launch_bounds__(BM_THREADS)
k_bm_get_decode(const uint8_t* __restrict__ enc, const uint8_t* __restrict__ desc,
                const GetMeta* __restrict__ meta, const uint32_t* __restrict__ values, uint64_t D,
                uint32_t* __restrict__ out, int* __restrict__ err) {
  __shared__ uint32_t ws[BM_THREADS / 32 + 2];
  __shared__ uint32_t s_runoff[2048 + 1];
  const GetMeta m = meta[blockIdx.x];
  const uint32_t key = ld16(desc + 4 * blockIdx.x);
  const uint8_t* pay = enc + m.pay;
  uint32_t* dst = out + m.out;
  auto emit = [&](uint32_t at, uint32_t low) {
    if (at >= m.card) {
      atomicMax(err, 1);
      return;
    }
    const uint32_t idx = (key << 16) | low;
    if ((uint64_t)idx >= D) {
      atomicMax(err, 2);  // "bitmask is out of bound", file/bitmask.go:41-44
      return;
    }
    dst[at] = __ldg(values + idx);
  };
  if (m.type == 0) {
    for (uint32_t k = threadIdx.x; k < m.card; k += BM_THREADS) emit(k, ld16(pay + 2 * k));
  } else if (m.type == 1) {
    constexpr uint32_t PER = 4096 / BM_THREADS;  // u16 pieces per thread, consecutive
    uint32_t piece[PER];
    uint32_t c = 0;
#pragma unroll
    for (uint32_t j = 0; j < PER; j++) {
      piece[j] = ld16(pay + 2 * (threadIdx.x * PER + j));
      c += __popc(piece[j]);
    }
    uint32_t tot;
    uint32_t at = block_exclusive_scan(c, ws, tot);
    if (threadIdx.x == 0 && tot != m.card) atomicMax(err, 1);
#pragma unroll
    for (uint32_t j = 0; j < PER; j++) {
      uint32_t x = piece[j];
      while (x) {
        const uint32_t b = __ffs(x) - 1;
        x &= x - 1;
        emit(at++, (threadIdx.x * PER + j) * 16 + b);
      }
    }
  } else {
    const uint32_t nr = ld16(pay);
    if (nr > 2048u) {  // more runs than a 65536-value chunk can hold
      if (threadIdx.x == 0) atomicMax(err, 1);
      return;
    }
    uint32_t run = 0;
    for (uint32_t base = 0; base < nr; base += BM_THREADS) {
      const uint32_t r = base + threadIdx.x;
      const uint32_t len = r < nr ? ld16(pay + 2 + 4 * r + 2) + 1 : 0u;
      uint32_t tot;
      const uint32_t ex = block_exclusive_scan(len, ws, tot);
      if (r < nr) s_runoff[r] = run + ex;
      run += tot;
    }
    if (threadIdx.x == 0) {
      s_runoff[nr] = run;
      if (run != m.card) atomicMax(err, 1);
    }
    __syncthreads();
    const uint32_t n = run < m.card ? run : m.card;
    for (uint32_t e = threadIdx.x; e < n; e += BM_THREADS) {
      uint32_t lo = 0, hi = nr;  // run holding element e
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (s_runoff[mid + 1] <= e)
          lo = mid + 1;
        else
          hi = mid;
      }
      emit(e, ld16(pay + 2 + 4 * lo) + (e - s_runoff[lo]));
    }
  }
}

int bm_reserve(ii2_bitmask* bm, uint64_t extra, cudaStream_t s) {
  const uint64_t need = bm->n + extra;
  if (need > bm->values_cap) {
    uint64_t cap = bm->values_cap ? bm->values_cap : 1024;
    while (cap < need) cap *= 2;
    DevBuf<uint32_t> nv;
    II2_TRY(nv.alloc(cap, s));
    if (bm->n)
      II2_CUDA_TRY(cudaMemcpyAsync(nv.p, bm->values.p, bm->n * 4, cudaMemcpyDeviceToDevice, s));
    bm->values = std::move(nv);
    bm->values_cap = cap;
  }
  if (2 * need + 2 > bm->table_cap) {
    uint64_t cap = 1024;
    while (cap < 4 * need + 4) cap *= 2;  // rebuilt at <= 25 % load, refilled up to 50 %
    DevBuf<unsigned long long> nt;
    II2_TRY(nt.alloc(cap, s));
    II2_CUDA_TRY(cudaMemsetAsync(nt.p, 0xFF, cap * 8, s));
    if (bm->n) {
      k_bm_build<<<div_up(bm->n, BM_THREADS), BM_THREADS, 0, s>>>(nt.p, cap - 1, bm->values.p, bm->n);
      II2_LAUNCHED();
    }
    bm->table = std::move(nt);
    bm->table_cap = cap;
  }
  return II2_OK;
}

// (Re)build the inverse if the dictionary allows it.  Synchronises the stream once (the maximum).
int bm_refresh_inverse(ii2_bitmask* bm, cudaStream_t s) {
  if (bm->inv_for_n == bm->n) return II2_OK;  // up to date (or known not to pay for this length)
  bm->inv_for_n = bm->n;
  bm->inv_len = 0;
  if (bm->n < 1024) return II2_OK;  // tiny dictionaries: the hash path is launch-bound anyway
  DevBuf<uint32_t> d_max;
  II2_TRY(d_max.alloc_scratch(1, s));
  II2_CUDA_TRY(cudaMemsetAsync(d_max.p, 0, 4, s));
  k_bm_max<<<(unsigned)std::min<uint64_t>(div_up(bm->n, BM_THREADS), 1184), BM_THREADS, 0, s>>>(
      bm->values.p, bm->n, d_max.p);
  II2_LAUNCHED();
  uint32_t* h = reinterpret_cast<uint32_t*>(pinned_scratch() + 28);
  II2_TRY(small_copy(h, d_max.p, 4, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  const uint64_t len = (uint64_t)h[0] + 1;
  if (len > 16 * bm->n + (1ull << 20) || len > (1ull << 30)) return II2_OK;  // too sparse
  II2_TRY(bm->inv.alloc(len, s));
  II2_CUDA_TRY(cudaMemsetAsync(bm->inv.p, 0xFF, len * 4, s));
  k_bm_inv_build<<<div_up(bm->n, BM_THREADS), BM_THREADS, 0, s>>>(bm->values.p, bm->n, bm->inv.p);
  II2_LAUNCHED();
  bm->inv_len = len;
  return II2_OK;
}

}  // namespace

extern "C" {

int ii2_bitmask_new(const uint32_t* init, uint64_t n, ii2_bitmask** out) {
  if (!out || (n && !init)) return II2_ERR_INVALID;
  *out = nullptr;
  II2_TRY(ctx_require());
  if (n >= 0xFFFFFFFEull) {
    set_last_error("bitmask dictionary of %llu values (indexes are uint32)", (unsigned long long)n);
    return II2_ERR_UNSUPPORTED;
  }
  cudaStream_t s = cur_stream();
  std::unique_ptr<ii2_bitmask> bm(new ii2_bitmask());
  II2_TRY(bm_reserve(bm.get(), n, s));
  if (n) II2_CUDA_TRY(cudaMemcpyAsync(bm->values.p, init, n * 4, cudaMemcpyHostToDevice, s));
  bm->n = n;
  // the table was sized for n but built over an empty dictionary: fill it now
  if (n) {
    k_bm_build<<<div_up(n, BM_THREADS), BM_THREADS, 0, s>>>(bm->table.p, bm->table_cap - 1,
                                                            bm->values.p, n);
    II2_LAUNCHED();
  }
  II2_TRY(bm_refresh_inverse(bm.get(), s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  arena_reset(s);
  *out = bm.release();
  return II2_OK;
}

void ii2_bitmask_free(ii2_bitmask* bm) {
  if (!bm) return;
  DeviceScope on(bm->device);
  delete bm;
}

int ii2_bitmask_all_values(const ii2_bitmask* bm, uint32_t** vals, uint64_t* n) {
  if (!bm || !vals || !n) return II2_ERR_INVALID;
  *vals = nullptr;
  *n = 0;
  II2_TRY(ctx_require_device(bm->device));
  cudaStream_t s = cur_stream();
  uint32_t* h = static_cast<uint32_t*>(pinned_alloc(bm->n * 4 + 4));
  if (!h) return II2_ERR_NOMEM;
  if (bm->n) {
    cudaError_t e = cudaMemcpyAsync(h, bm->values.p, bm->n * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
      pinned_free(h);
      set_last_error("all_values copy: %s", cudaGetErrorString(e));
      return II2_ERR_CUDA;
    }
  }
  *vals = h;
  *n = bm->n;
  return II2_OK;
}

int ii2_bitmask_put(ii2_bitmask* bm, const uint32_t* vals, uint64_t n, uint8_t** bytes,
                    uint64_t* nbytes) {
  if (!bm || !bytes || !nbytes || (n && !vals)) return II2_ERR_INVALID;
  *bytes = nullptr;
  *nbytes = 0;
  II2_TRY(ctx_require_device(bm->device));
  if (bm->n + n >= 0xFFFFFFFEull) {
    set_last_error("bitmask dictionary would exceed uint32 indexes");
    return II2_ERR_UNSUPPORTED;
  }
  cudaStream_t s = cur_stream();
  ProfScope scope("k3b_put", s);
  II2_TRY(bm_reserve(bm, n, s));
  const uint32_t D = (uint32_t)bm->n;
  const uint64_t mask = bm->table_cap - 1;
  const uint64_t max_bits = bm->n + n;
  const uint32_t nchunks = (uint32_t)((max_bits + 65535) / 65536);
  DevBuf<uint32_t> d_vals, d_bits, d_card, d_cidx, d_cont;
  DevBuf<uint64_t> d_rank, d_poff, d_tot;
  II2_TRY(d_vals.alloc_scratch(n, s));
  II2_TRY(d_rank.alloc_scratch(n + 1, s));
  II2_TRY(d_bits.alloc_scratch((size_t)(nchunks ? nchunks : 1) * CHUNK_WORDS, s));
  II2_TRY(d_card.alloc_scratch(nchunks ? nchunks : 1, s));
  II2_TRY(d_cidx.alloc_scratch(nchunks ? nchunks : 1, s));
  II2_TRY(d_cont.alloc_scratch(nchunks ? nchunks : 1, s));
  II2_TRY(d_poff.alloc_scratch(nchunks ? nchunks : 1, s));
  II2_TRY(d_tot.alloc_scratch(4, s));
  II2_CUDA_TRY(cudaMemsetAsync(d_bits.p, 0, (size_t)(nchunks ? nchunks : 1) * CHUNK_WORDS * 4, s));
  uint64_t h_tot[4] = {0, 0, 0, 0};
  bool direct = false;
  if (n) II2_CUDA_TRY(cudaMemcpyAsync(d_vals.p, vals, n * 4, cudaMemcpyHostToDevice, s));
  ProfScope kscope("k3b_put_kernels", s);  // values resident -> serialised bitmap resident
  if (n && bm->inv_len && bm->inv_for_n == bm->n && n >= 1024) {
    // every value already in the dictionary (the usual Put over a known id universe): one probe
    // of the direct-address inverse per value; a miss means appends, which the general path
    // orders (first occurrence, input order)
    DevBuf<uint32_t> d_miss;
    II2_TRY(d_miss.alloc_scratch(1, s));
    II2_CUDA_TRY(cudaMemsetAsync(d_miss.p, 0, 4, s));
    k_bm_put_direct<<<div_up(n, BM_THREADS), BM_THREADS, 0, s>>>(bm->inv.p, bm->inv_len, d_vals.p, n,
                                                                 d_bits.p, d_miss.p);
    II2_LAUNCHED();
    uint32_t* h_miss = reinterpret_cast<uint32_t*>(pinned_scratch() + 29);
    II2_TRY(small_copy(h_miss, d_miss.p, 4, s));
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    direct = h_miss[0] == 0;
    if (direct)
      II2_CUDA_TRY(cudaMemsetAsync(d_tot.p + 3, 0, 8, s));  // nothing appended
    else
      II2_CUDA_TRY(cudaMemsetAsync(d_bits.p, 0, (size_t)(nchunks ? nchunks : 1) * CHUNK_WORDS * 4, s));
  }
  if (n && !direct) {
    const unsigned g = div_up(n, BM_THREADS), g1 = div_up(n + 1, BM_THREADS);
    k_bm_put_insert<<<g, BM_THREADS, 0, s>>>(bm->table.p, mask, d_vals.p, n, D);
    II2_LAUNCHED();
    k_bm_put_flag<<<g1, BM_THREADS, 0, s>>>(bm->table.p, mask, d_vals.p, n, D, d_rank.p);
    II2_LAUNCHED();
    II2_TRY(exclusive_scan_u64(d_rank.p, n + 1, d_tot.p + 3, s));
    k_bm_put_resolve<<<g, BM_THREADS, 0, s>>>(bm->table.p, mask, d_vals.p, n, D, d_rank.p,
                                              bm->values.p, d_bits.p);
    II2_LAUNCHED();
    k_bm_put_fixup<<<g, BM_THREADS, 0, s>>>(bm->table.p, mask, d_vals.p, n, D, d_rank.p);
    II2_LAUNCHED();
  } else if (!n) {
    II2_CUDA_TRY(cudaMemsetAsync(d_tot.p + 3, 0, 8, s));
  }
  if (nchunks) {
    k_bm_chunk_card<<<nchunks, BM_THREADS, 0, s>>>(d_bits.p, d_card.p);
    II2_LAUNCHED();
  }
  k_bm_chunk_scan<<<1, 1024, 0, s>>>(d_card.p, nchunks, d_cidx.p, d_poff.p, d_cont.p, d_tot.p);
  II2_LAUNCHED();
  II2_CUDA_TRY(cudaMemcpyAsync(h_tot, d_tot.p, 32, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  bm->n += h_tot[3];  // appended dictionary entries (the inverse is rebuilt by the next call)
  if (h_tot[3]) II2_TRY(bm_refresh_inverse(bm, s));
  const uint32_t nc = (uint32_t)h_tot[0];
  const int has_run = h_tot[2] != 0;
  const int has_off = !has_run || nc >= 4;  // noOffsetThreshold
  const uint32_t desc_at = has_run ? 4 + (nc + 7) / 8 : 8;
  const uint32_t offs_at = desc_at + 4 * nc;
  const uint64_t data_at = offs_at + (has_off ? 4ull * nc : 0ull);
  const uint64_t total = data_at + h_tot[1];
  if (total >= (1ull << 32)) {
    set_last_error("serialised bitmap exceeds 4 GiB");
    return II2_ERR_UNSUPPORTED;
  }
  DevBuf<uint8_t> d_out;
  II2_TRY(d_out.alloc_scratch(total, s, 8));
  k_bm_header<<<div_up((uint64_t)nc + 1, BM_THREADS), BM_THREADS, 0, s>>>(
      d_card.p, d_poff.p, d_cont.p, nc, has_run, d_out.p, desc_at, offs_at, has_off,
      (uint32_t)data_at);
  II2_LAUNCHED();
  if (nc) {
    k_bm_payload<<<nc, BM_THREADS, 0, s>>>(d_bits.p, d_card.p, d_poff.p, d_cont.p, d_out.p,
                                           (uint32_t)data_at);
    II2_LAUNCHED();
  }
  kscope.end();
  uint8_t* h = static_cast<uint8_t*>(pinned_alloc(total + 8));
  if (!h) return II2_ERR_NOMEM;
  cudaError_t e = cudaMemcpyAsync(h, d_out.p, total, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    pinned_free(h);
    set_last_error("bitmask put: %s", cudaGetErrorString(e));
    return II2_ERR_CUDA;
  }
  arena_reset(s);
  *bytes = h;
  *nbytes = total;
  return II2_OK;
}

int ii2_bitmask_get(const ii2_bitmask* bm, const uint8_t* enc, uint64_t nenc, uint32_t** vals,
                    uint64_t* n) {
  if (!bm || !vals || !n || (nenc && !enc)) return II2_ERR_INVALID;
  *vals = nullptr;
  *n = 0;
  II2_TRY(ctx_require_device(bm->device));
  cudaStream_t s = cur_stream();
  ProfScope scope("k3b_get", s);
  const uint32_t meta_cap = (uint32_t)std::min<uint64_t>(65536, nenc / 4 + 1);
  DevBuf<uint8_t> d_enc;
  DevBuf<GetMeta> d_meta;
  DevBuf<uint64_t> d_info;
  DevBuf<int> d_err;
  II2_TRY(d_enc.alloc_scratch(nenc, s, 16));
  II2_TRY(d_meta.alloc_scratch(meta_cap, s));
  II2_TRY(d_info.alloc_scratch(3, s));
  II2_TRY(d_err.alloc_scratch(1, s));
  if (nenc) II2_CUDA_TRY(cudaMemcpyAsync(d_enc.p, enc, nenc, cudaMemcpyHostToDevice, s));
  II2_CUDA_TRY(cudaMemsetAsync(d_err.p, 0, 4, s));
  ProfScope kscope("k3b_get_kernels", s);  // bytes resident -> values resident
  k_bm_get_parse<<<1, 1024, 0, s>>>(d_enc.p, nenc, d_meta.p, meta_cap, d_info.p);
  II2_LAUNCHED();
  uint64_t info[3] = {0, 0, 0};
  II2_CUDA_TRY(cudaMemcpyAsync(info, d_info.p, 24, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  if (info[2]) {
    set_last_error("undecodable roaring buffer");
    return II2_ERR_CORRUPT;
  }
  const uint32_t nc = (uint32_t)info[0];
  const uint64_t total = info[1];
  DevBuf<uint32_t> d_out;
  II2_TRY(d_out.alloc_scratch(total, s));
  if (nc) {
    const uint32_t cookie = (uint32_t)enc[0] | ((uint32_t)enc[1] << 8);
    const uint64_t desc_at = cookie == 12347u ? 4 + ((uint64_t)nc + 7) / 8 : 8;
    k_bm_get_decode<<<nc, BM_THREADS, 0, s>>>(d_enc.p, d_enc.p + desc_at, d_meta.p, bm->values.p,
                                              bm->n, d_out.p, d_err.p);
    II2_LAUNCHED();
  }
  kscope.end();
  II2_CUDA_TRY(cudaMemcpyAsync(pinned_scratch() + 27, d_err.p, 4, cudaMemcpyDeviceToHost, s));
  uint32_t* h = static_cast<uint32_t*>(pinned_alloc(total * 4 + 4));
  if (!h) return II2_ERR_NOMEM;
  cudaError_t e = cudaSuccess;
  if (total) e = cudaMemcpyAsync(h, d_out.p, total * 4, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  const int herr = *reinterpret_cast<const int*>(pinned_scratch() + 27);
  if (e != cudaSuccess) {
    pinned_free(h);
    set_last_error("bitmask get: %s", cudaGetErrorString(e));
    return II2_ERR_CUDA;
  }
  if (herr) {
    pinned_free(h);
    if (herr == 2) {
      set_last_error("bitmask is out of bound: index beyond the %llu-value dictionary",
                     (unsigned long long)bm->n);
      return II2_ERR_BITMASK_OOB;
    }
    set_last_error("undecodable roaring buffer");
    return II2_ERR_CORRUPT;
  }
  arena_reset(s);
  *vals = h;
  *n = total;
  return II2_OK;
}

}  // extern "C"
