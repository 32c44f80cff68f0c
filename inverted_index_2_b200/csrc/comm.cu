// comm.cu — the cross-shard exchange behind the C-ABI (include/ii2.h, "cross-shard exchange").
//
// Replaces, when the shards of one index live on several GPUs (one process per GPU, contiguous
// shard-key ranges per rank, so rank order == term order):
//   - the ordered concatenation of shard streams of InvertedIndex.Read
//     (inverted_index.go:330-338): ii2_read_gather — ONE all-gather of a 32-byte size record,
//     ONE group of ncclSend / ncclRecv that moves the four flat arrays of every rank straight
//     from its result to their final place on the root, and one kernel that rebases the offsets;
//   - the union of the per-shard maps of PrefixSearch under its mutex + the final slices.Sort /
//     slices.Compact (inverted_index.go:274-292): ii2_prefix_gather — the per-prefix value lists
//     of every rank land back to back on the root and the heavy-term union kernels
//     (k12_union.cu, sort forced) make every prefix sorted-unique again.
// Compaction itself needs no exchange: shards never interact (shard.go:19-20).
//
// The same two operations inside ONE process that drives several GPUs (ii2_init with a device
// set): ii2_read_gather_devices — one kernel on the root device reads every part's arrays
// straight from peer HBM (peer access over NVLink) and writes them, offsets rebased, to their
// final place; ii2_prefix_gather_devices — the same union on the root as ii2_prefix_gather.
//
// NCCL is bound at run time (dlopen of libnccl.so.2): the library must load on hosts without
// it, and inside a process that already carries torch's NCCL the same instance is reused.
#include <dlfcn.h>
#include <nccl.h>

#include <memory>
#include <mutex>
#include <vector>

#include "handles.cuh"

namespace {

struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*);
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
  ncclResult_t (*CommDestroy)(ncclComm_t);
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*GroupStart)();
  ncclResult_t (*GroupEnd)();
  const char* (*GetErrorString)(ncclResult_t);
  bool ok = false;
};

NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return;
    bool all = true;
    auto sym = [&](const char* name) -> void* {
      void* p = dlsym(h, name);
      if (!p) all = false;
      return p;
    };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
    api.Send = reinterpret_cast<decltype(api.Send)>(sym("ncclSend"));
    api.Recv = reinterpret_cast<decltype(api.Recv)>(sym("ncclRecv"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    api.ok = all;
  });
  return api;
}

struct Comm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
};
Comm g_comm;
std::mutex g_comm_mu;

#define II2_NCCL_TRY(expr)                                                              \
  do {                                                                                  \
    ncclResult_t _r = (expr);                                                           \
    if (_r != ncclSuccess) {                                                            \
      set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, nccl().GetErrorString(_r)); \
      return II2_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

constexpr int kMaxWorld = 64;

// The ordered concatenation of up to kMaxWorld read results: part r's four arrays go to the
// output at the bases T[r] (terms), TB[r] (term bytes), P[r] (postings), its offsets shifted by
// TB[r] / P[r]; the terminal entries close the arrays.  `src` may point into peer HBM (in-process
// gather) or at the destination itself (NCCL gather: the pieces were received in place and only
// the offsets still need their base).
struct GatherPart {
  const uint8_t* tb;
  const uint32_t* toff;  // [T_r] (the part's terminal entry is not read)
  const uint32_t* post;
  const uint64_t* poff;  // [T_r]
};
struct GatherArgs {
  GatherPart src[kMaxWorld];
  uint8_t* tb;
  uint32_t* toff;
  uint32_t* post;
  uint64_t* poff;
  uint64_t T[kMaxWorld + 1], TB[kMaxWorld + 1], P[kMaxWorld + 1];
  int world;
};

// n elements (4 or 8 bytes) from src to dst plus `add`, by the threads t of nt: the few elements
// before dst's first 16-byte boundary, then 16-byte stores (16-byte loads when src has the same
// phase, element loads otherwise), then the rest.  src == dst is allowed (in-place rebase).
template <typename E>
__device__ __forceinline__ void gather_copy_add(const E* src, E* dst, uint64_t n, E add, uint64_t t,
                                                uint64_t nt) {
  constexpr int kPer = 16 / sizeof(E);
  if (src == dst && add == 0) return;
  const uint64_t lead = ((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15) / sizeof(E);
  const uint64_t head = lead < n ? lead : n;
  if (t < head) dst[t] = src[t] + add;
  const E* s = src + head;
  E* d = dst + head;
  const uint64_t body = (n - head) / kPer;
  const bool s16 = (reinterpret_cast<uintptr_t>(s) & 15) == 0;
  for (uint64_t v = t; v < body; v += nt) {
    E x[kPer];
    if (s16) {
      const uint4 q = reinterpret_cast<const uint4*>(s)[v];
      memcpy(x, &q, 16);
    } else {
#pragma unroll
      for (int k = 0; k < kPer; k++) x[k] = s[v * kPer + k];
    }
#pragma unroll
    for (int k = 0; k < kPer; k++) x[k] += add;
    uint4 q;
    memcpy(&q, x, 16);
    reinterpret_cast<uint4*>(d)[v] = q;
  }
  const uint64_t done = head + body * kPer;
  if (t < n - done) dst[done + t] = src[done + t] + add;
}

// n bytes from src to dst; both may start at any address (a part's term bytes land at an
// arbitrary offset of the output).  16-byte stores at dst's boundaries; a source of another
// phase is read as aligned words and funnel-shifted into place.
__device__ __forceinline__ void gather_copy_bytes(const uint8_t* src, uint8_t* dst, uint64_t n, uint64_t t,
                                                  uint64_t nt) {
  if (src == dst) return;
  const uint64_t lead = (16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15;
  const uint64_t head = lead < n ? lead : n;
  if (t < head) dst[t] = src[t];
  const uint8_t* s = src + head;
  uint8_t* d = dst + head;
  const uint64_t body = (n - head) >> 4;
  const unsigned sh = (unsigned)(reinterpret_cast<uintptr_t>(s) & 3);
  const bool s16 = (reinterpret_cast<uintptr_t>(s) & 15) == 0;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(s - sh);
  for (uint64_t v = t; v < body; v += nt) {
    uint4 q;
    if (s16) {
      q = reinterpret_cast<const uint4*>(s)[v];
    } else {
      const uint32_t* p = w + 4 * v;
      const uint32_t a0 = p[0], a1 = p[1], a2 = p[2], a3 = p[3];
      if (sh) {  // the 5th word holds the vector's last bytes: never past the source's last word
        const uint32_t a4 = p[4];
        q.x = __funnelshift_r(a0, a1, 8 * sh);
        q.y = __funnelshift_r(a1, a2, 8 * sh);
        q.z = __funnelshift_r(a2, a3, 8 * sh);
        q.w = __funnelshift_r(a3, a4, 8 * sh);
      } else {
        q = make_uint4(a0, a1, a2, a3);
      }
    }
    reinterpret_cast<uint4*>(d)[v] = q;
  }
  const uint64_t done = head + (body << 4);
  if (t < n - done) dst[done + t] = src[done + t];
}

// grid (x, part, array): blockIdx.z picks the array (0 term bytes, 1 term_off, 2 postings,
// 3 post_off) of part blockIdx.y; the x CTAs of the pair stride over it.
__global__ void __launch_bounds__(256) k_gather_parts(const GatherArgs a) {
  const int r = blockIdx.y;
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t nt = (uint64_t)gridDim.x * blockDim.x;
  const GatherPart& g = a.src[r];
  const uint64_t T = r < a.world ? a.T[r + 1] - a.T[r] : 0;
  if (r < a.world) switch (blockIdx.z) {
    case 0: gather_copy_bytes(g.tb, a.tb + a.TB[r], a.TB[r + 1] - a.TB[r], t, nt); break;
    case 1: gather_copy_add<uint32_t>(g.toff, a.toff + a.T[r], T, (uint32_t)a.TB[r], t, nt); break;
    case 2: gather_copy_add<uint32_t>(g.post, a.post + a.P[r], a.P[r + 1] - a.P[r], 0u, t, nt); break;
    default: gather_copy_add<uint64_t>(g.poff, a.poff + a.T[r], T, a.P[r], t, nt); break;
  }
  if (r == 0 && blockIdx.z == 0 && t == 0) {
    const int W = a.world;
    a.toff[a.T[W]] = (uint32_t)a.TB[W];
    a.poff[a.T[W]] = a.P[W];
  }
}

int launch_gather_parts(const GatherArgs& a, cudaStream_t s) {
  const int W = a.world;
  uint64_t most = 1;  // 16-byte vectors of the largest array piece
  for (int r = 0; r < W; r++) {
    const uint64_t T = a.T[r + 1] - a.T[r];
    most = std::max<uint64_t>(most, std::max<uint64_t>((a.TB[r + 1] - a.TB[r]) / 16,
                                                        std::max<uint64_t>(T / 2, (a.P[r + 1] - a.P[r]) / 4)));
  }
  const unsigned gx = (unsigned)std::min<uint64_t>(256, div_up(most, 256 * 4));
  k_gather_parts<<<dim3(gx, (unsigned)std::max(W, 1), 4), 256, 0, s>>>(a);
  II2_LAUNCHED();
  return II2_OK;
}

// one (prefix, rank) source of the union on the root: where rank r's values of prefix p landed
__global__ void __launch_bounds__(256)
k_prefix_sources(const uint64_t* __restrict__ voff_all /* [world][np+1] */, const uint32_t* __restrict__ vals,
                 const uint64_t* __restrict__ vbase /* [world] */, uint32_t np, int world,
                 uint64_t* __restrict__ src_ptr, uint32_t* __restrict__ src_len, GroupIn* __restrict__ gin,
                 uint32_t* __restrict__ rec, uint32_t* __restrict__ flags) {
  const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (uint64_t)np * world) return;
  const uint32_t p = (uint32_t)(id / world);
  const int r = (int)(id % world);
  const uint64_t* vo = voff_all + (uint64_t)r * (np + 1);
  uint64_t len = vo[p + 1] - vo[p];
  if (len > 0xFFFFFFFFull) {
    atomicExch(&flags[0], 1u);
    len = 0;
  }
  src_ptr[id] = reinterpret_cast<uint64_t>(vals + vbase[r] + vo[p]);
  src_len[id] = (uint32_t)len;
  if (r == 0) {
    GroupIn g;
    g.inst = 0;
    g.tlen = 0;
    g.src = (uint32_t)id;
    g.c = (uint32_t)world;
    g.L = 0xFFFFFFFFu;
    g.pst = 0;
    g.eslot = 0;
    g.pad = 0;
    gin[p] = g;
    rec[p] = p;
  }
}

__global__ void __launch_bounds__(256)
k_prefix_counts(const GroupRec* __restrict__ recs, uint32_t np, uint64_t* __restrict__ cnt) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < np) cnt[p] = recs[p].cnt;
  if (p == np) cnt[np] = 0;
}

__global__ void __launch_bounds__(256)
k_prefix_place(const GroupRec* __restrict__ recs, const uint64_t* __restrict__ off,
               uint32_t* __restrict__ out) {
  const GroupRec r = recs[blockIdx.y];
  const uint32_t* src = reinterpret_cast<const uint32_t*>(r.dec);
  uint32_t* dst = out + off[blockIdx.y];
  for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < r.cnt; i += (uint64_t)gridDim.x * 256)
    dst[i] = src[i];
}

__global__ void __launch_bounds__(256)
k_or_matched(const uint8_t* __restrict__ all /* [world][np] */, uint32_t np, int world,
             uint8_t* __restrict__ out) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= np) return;
  uint8_t m = 0;
  for (int r = 0; r < world; r++) m |= all[(uint64_t)r * np + p];
  out[p] = m ? 1 : 0;
}

int comm_ready() {
  if (!g_comm.comm) {
    set_last_error("ii2_comm_init has not been called");
    return II2_ERR_INVALID;
  }
  return II2_OK;
}

int read_gather_impl(const ii2_result* local, int root, ii2_result** out, cudaStream_t s) {
  NcclApi& n = nccl();
  const int world = g_comm.world, rank = g_comm.rank;
  const bool recv = root < 0 || rank == root;
  // ---- sizes of every rank: one all-gather of {terms, term bytes, postings, -}
  DevBuf<uint64_t> d_sz;
  II2_TRY(d_sz.alloc_scratch(4 * (size_t)(world + 1), s));
  PinnedBlock h_blk(8 * 4 * (size_t)(world + 1));
  uint64_t* h = static_cast<uint64_t*>(h_blk.p);
  if (!h) return II2_ERR_NOMEM;
  uint64_t* mine = h + 4 * (size_t)world;
  mine[0] = local->T;
  mine[1] = local->TB;
  mine[2] = local->P;
  mine[3] = 0;
  II2_TRY(small_copy(d_sz.p + 4 * (size_t)world, mine, 32, s));
  II2_NCCL_TRY(n.AllGather(d_sz.p + 4 * (size_t)world, d_sz.p, 4, ncclUint64, g_comm.comm, s));
  II2_TRY(small_copy(h, d_sz.p, 32 * (size_t)world, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  GatherArgs b;
  b.world = world;
  b.T[0] = b.TB[0] = b.P[0] = 0;
  for (int r = 0; r < world; r++) {
    b.T[r + 1] = b.T[r] + h[4 * r];
    b.TB[r + 1] = b.TB[r] + h[4 * r + 1];
    b.P[r + 1] = b.P[r] + h[4 * r + 2];
  }
  if (b.TB[world] >= (1ull << 32) || b.T[world] >= 0xFFFFFFFFull) {
    set_last_error("gathered read exceeds 4 GiB of term bytes / 2^32-2 terms");
    return II2_ERR_UNSUPPORTED;
  }
  std::unique_ptr<ii2_result> res(new ii2_result());
  res->stream = s;
  res->has_dec = true;
  EmitOut& o = res->out;
  if (recv) {
    res->T = b.T[world];
    res->TB = b.TB[world];
    res->P = b.P[world];
    II2_TRY(o.term_bytes.alloc(res->TB, s, 32));
    II2_TRY(o.term_off.alloc(res->T + 1, s, 16));
    II2_TRY(o.post.alloc(res->P, s, 16));
    II2_TRY(o.post_off.alloc(res->T + 1, s, 16));
  } else {
    II2_TRY(o.term_bytes.alloc(0, s, 32));
    II2_TRY(o.term_off.alloc(1, s));
    II2_TRY(o.post.alloc(0, s));
    II2_TRY(o.post_off.alloc(1, s));
    II2_CUDA_TRY(cudaMemsetAsync(o.term_off.p, 0, 4, s));
    II2_CUDA_TRY(cudaMemsetAsync(o.post_off.p, 0, 8, s));
  }
  // ---- one exchange: every array of every rank straight to its final place
  const EmitOut& l = local->out;
  auto put = [&](int r, const void* src, void* dst, uint64_t bytes) -> int {  // rank r's piece
    if (!bytes) return II2_OK;
    if (r == rank) {
      if (recv) II2_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
      return II2_OK;
    }
    II2_NCCL_TRY(n.Recv(dst, bytes, ncclUint8, r, g_comm.comm, s));
    return II2_OK;
  };
  II2_NCCL_TRY(n.GroupStart());  // (closed below whatever happens inside: an open group poisons the communicator)
  int rc = II2_OK;
  for (int dst_rank = 0; dst_rank < world && rc == II2_OK; dst_rank++) {
    if (!(root < 0 || dst_rank == root) || dst_rank == rank) continue;
    // my pieces to the receiving rank (the same order on both sides)
    const uint64_t T = local->T;
    auto send = [&](const void* p, uint64_t bytes) -> int {
      if (!bytes) return II2_OK;
      II2_NCCL_TRY(n.Send(p, bytes, ncclUint8, dst_rank, g_comm.comm, s));
      return II2_OK;
    };
    if (rc == II2_OK) rc = send(l.term_bytes.p, local->TB);
    if (rc == II2_OK) rc = send(l.term_off.p, T * 4);
    if (rc == II2_OK) rc = send(l.post.p, local->P * 4);
    if (rc == II2_OK) rc = send(l.post_off.p, T * 8);
  }
  if (recv) {
    for (int r = 0; r < world && rc == II2_OK; r++) {
      const uint64_t T = h[4 * r], TBr = h[4 * r + 1], Pr = h[4 * r + 2];
      const bool me = r == rank;
      if (rc == II2_OK) rc = put(r, me ? l.term_bytes.p : nullptr, o.term_bytes.p + b.TB[r], TBr);
      if (rc == II2_OK) rc = put(r, me ? l.term_off.p : nullptr, o.term_off.p + b.T[r], T * 4);
      if (rc == II2_OK) rc = put(r, me ? l.post.p : nullptr, o.post.p + b.P[r], Pr * 4);
      if (rc == II2_OK) rc = put(r, me ? l.post_off.p : nullptr, o.post_off.p + b.T[r], T * 8);
    }
  }
  {
    const ncclResult_t ge = n.GroupEnd();
    II2_TRY(rc);
    II2_NCCL_TRY(ge);
  }
  if (recv) {  // the pieces landed in place: the offsets get their bases, the terminal entries
    b.tb = o.term_bytes.p;
    b.toff = o.term_off.p;
    b.post = o.post.p;
    b.poff = o.post_off.p;
    for (int r = 0; r < world; r++)
      b.src[r] = {b.tb + b.TB[r], b.toff + b.T[r], b.post + b.P[r], b.poff + b.T[r]};
    II2_TRY(launch_gather_parts(b, s));
  }
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  *out = res.release();
  return II2_OK;
}

int prefix_out_empty(uint32_t np, ii2_prefix_out* out);
int prefix_union_on_root(const uint64_t* d_voff, const uint32_t* d_vals, const uint8_t* d_m,
                         const std::vector<uint64_t>& vbase, uint32_t np, int world, ii2_prefix_out* out,
                         cudaStream_t s);

int prefix_gather_impl(const ii2_prefix_out* local, int root, ii2_prefix_out* out, cudaStream_t s) {
  NcclApi& n = nccl();
  const int world = g_comm.world, rank = g_comm.rank;
  const bool recv = root < 0 || rank == root;
  const uint32_t np = (uint32_t)local->n_prefixes;
  const uint64_t nv = np ? local->value_off[np] : 0;
  // ---- every rank's value offsets and matched flags: fixed size, two all-gathers
  DevBuf<uint64_t> d_voff;
  DevBuf<uint8_t> d_m;
  const size_t row = (size_t)np + 1;
  II2_TRY(d_voff.alloc_scratch(row * (size_t)(world + 1), s));
  II2_TRY(d_m.alloc_scratch(((size_t)np + 16) * (size_t)(world + 1), s));
  PinnedBlock voff_blk(8 * row * (size_t)world + 64);
  uint64_t* h_voff = static_cast<uint64_t*>(voff_blk.p);
  if (!h_voff) return II2_ERR_NOMEM;
  uint64_t* my_voff = d_voff.p + row * (size_t)world;
  uint8_t* my_m = d_m.p + (size_t)np * world;
  if (np) {
    II2_CUDA_TRY(cudaMemcpyAsync(my_voff, local->value_off, row * 8, cudaMemcpyHostToDevice, s));
    II2_CUDA_TRY(cudaMemcpyAsync(my_m, local->matched, np, cudaMemcpyHostToDevice, s));
  } else {
    II2_CUDA_TRY(cudaMemsetAsync(my_voff, 0, 8, s));
  }
  II2_NCCL_TRY(n.AllGather(my_voff, d_voff.p, row, ncclUint64, g_comm.comm, s));
  if (np) II2_NCCL_TRY(n.AllGather(my_m, d_m.p, np, ncclUint8, g_comm.comm, s));
  II2_CUDA_TRY(cudaMemcpyAsync(h_voff, d_voff.p, 8 * row * (size_t)world, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  std::vector<uint64_t> vbase(world + 1, 0);
  for (int r = 0; r < world; r++) vbase[r + 1] = vbase[r] + h_voff[row * r + np];
  // ---- the values: one group of sends / receives, rank r's block at vbase[r]
  DevBuf<uint32_t> d_vals, d_mine;
  II2_TRY(d_vals.alloc_scratch(recv ? vbase[world] : 0, s));
  II2_TRY(d_mine.alloc_scratch(nv, s));
  if (nv) II2_CUDA_TRY(cudaMemcpyAsync(d_mine.p, local->values, nv * 4, cudaMemcpyHostToDevice, s));
  II2_NCCL_TRY(n.GroupStart());
  {
    int rc = II2_OK;
    auto xfer = [&](bool send, void* p, uint64_t bytes, int peer) -> int {
      if (send)
        II2_NCCL_TRY(n.Send(p, bytes, ncclUint8, peer, g_comm.comm, s));
      else
        II2_NCCL_TRY(n.Recv(p, bytes, ncclUint8, peer, g_comm.comm, s));
      return II2_OK;
    };
    for (int dst_rank = 0; dst_rank < world && rc == II2_OK; dst_rank++) {
      if (!(root < 0 || dst_rank == root) || dst_rank == rank || !nv) continue;
      rc = xfer(true, d_mine.p, nv * 4, dst_rank);
    }
    if (recv) {
      for (int r = 0; r < world && rc == II2_OK; r++) {
        const uint64_t cnt = vbase[r + 1] - vbase[r];
        if (!cnt) continue;
        if (r == rank) {
          if (cudaMemcpyAsync(d_vals.p + vbase[r], d_mine.p, cnt * 4, cudaMemcpyDeviceToDevice, s) != cudaSuccess) {
            set_last_error("prefix gather: local copy failed");
            rc = II2_ERR_CUDA;
          }
        } else {
          rc = xfer(false, d_vals.p + vbase[r], cnt * 4, r);
        }
      }
    }
    const ncclResult_t ge = n.GroupEnd();  // always closed
    II2_TRY(rc);
    II2_NCCL_TRY(ge);
  }
  if (!recv || np == 0) {
    II2_CUDA_TRY(cudaStreamSynchronize(s));
    return prefix_out_empty(np, out);
  }
  return prefix_union_on_root(d_voff.p, d_vals.p, d_m.p, vbase, np, world, out, s);
}

// ii2_prefix_out of n_prefixes = np with no match (a non-root rank, or no prefix at all).
int prefix_out_empty(uint32_t np, ii2_prefix_out* out) {
  std::unique_ptr<HostOwner> own(new HostOwner());
  out->n_prefixes = np;
  out->matched = own->alloc<uint8_t>((size_t)np + 1);
  out->value_off = own->alloc<uint64_t>((size_t)np + 1);
  out->values = own->alloc<uint32_t>(0);
  if (!out->matched || !out->value_off || !out->values) return II2_ERR_NOMEM;
  memset(out->matched, 0, (size_t)np + 1);
  memset(out->value_off, 0, ((size_t)np + 1) * 8);
  out->_owner = own.release();
  return II2_OK;
}

// The union half of both prefix gathers, on the root device: `world` prefix outputs of the same
// np (> 0) prefixes have landed there — value offsets d_voff [world][np+1] (relative to the part),
// values d_vals with part r's block at vbase[r], matched flags d_m [world][np].  Per prefix, the
// sorted-unique union of the parts' lists (inverted_index.go:289-292) and the OR of the flags,
// downloaded into `out`.
int prefix_union_on_root(const uint64_t* d_voff, const uint32_t* d_vals, const uint8_t* d_m,
                         const std::vector<uint64_t>& vbase, uint32_t np, int world, ii2_prefix_out* out,
                         cudaStream_t s) {
  const size_t row = (size_t)np + 1;
  std::unique_ptr<HostOwner> own(new HostOwner());
  out->n_prefixes = np;
  out->matched = own->alloc<uint8_t>((size_t)np + 1);
  out->value_off = own->alloc<uint64_t>(row);
  if (!out->matched || !out->value_off) return II2_ERR_NOMEM;
  // ---- per prefix: the sorted-unique union of its `world` lists (inverted_index.go:289-292)
  const uint64_t pairs = (uint64_t)np * world;
  DevBuf<uint64_t> src_ptr, d_vbase, d_off, d_tot;
  DevBuf<uint32_t> src_len, rec, flags, large_tmp, large_enc;
  DevBuf<GroupIn> gin;
  DevBuf<GroupRec> recs;
  DevBuf<uint8_t> d_mout;
  II2_TRY(src_ptr.alloc_scratch(pairs, s));
  II2_TRY(src_len.alloc_scratch(pairs, s));
  II2_TRY(rec.alloc_scratch(np, s));
  II2_TRY(flags.alloc_scratch(2, s));
  II2_TRY(gin.alloc_scratch(np, s));
  II2_TRY(recs.alloc_scratch(np, s));
  II2_TRY(d_vbase.alloc_scratch(world + 1, s));
  II2_TRY(d_off.alloc_scratch(row, s));
  II2_TRY(d_tot.alloc_scratch(1, s));
  II2_TRY(d_mout.alloc_scratch(np, s));
  II2_CUDA_TRY(cudaMemsetAsync(flags.p, 0, 8, s));
  PinnedBlock small_blk(8 * (size_t)(world + 4));
  uint64_t* h_small = static_cast<uint64_t*>(small_blk.p);
  if (!h_small) return II2_ERR_NOMEM;
  for (int r = 0; r <= world; r++) h_small[r] = vbase[r];
  II2_TRY(small_copy(d_vbase.p, h_small, 8 * (size_t)(world + 1), s));
  k_prefix_sources<<<div_up(pairs, 256), 256, 0, s>>>(d_voff, d_vals, d_vbase.p, np, world, src_ptr.p,
                                                      src_len.p, gin.p, rec.p, flags.p);
  II2_LAUNCHED();
  LargeArgs la;
  la.rec = rec.p;
  la.bucket = nullptr;
  la.gin = gin.p;
  la.src_ptr = src_ptr.p;
  la.src_len = src_len.p;
  la.recs = recs.p;
  la.rem = RemovedSet{};
  la.want_enc = 0;
  la.keep_empty = 1;
  la.always_sort = 1;
  la.presorted = nullptr;
  la.bk_raw = nullptr;
  la.nb1 = 0;
  II2_TRY(k2_large_run(la, np, large_tmp, large_enc, s));
  k_prefix_counts<<<div_up((uint64_t)np + 1, 256), 256, 0, s>>>(recs.p, np, d_off.p);
  II2_LAUNCHED();
  II2_TRY(exclusive_scan_u64(d_off.p, row, d_tot.p, s));
  k_or_matched<<<div_up(np, 256), 256, 0, s>>>(d_m, np, world, d_mout.p);
  II2_LAUNCHED();
  II2_TRY(small_copy(h_small, d_tot.p, 8, s));
  II2_TRY(small_copy(h_small + 1, flags.p, 8, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  if ((uint32_t)h_small[1]) {
    set_last_error("prefix gather: one part holds more than 2^32-1 values under a prefix");
    return II2_ERR_UNSUPPORTED;
  }
  const uint64_t total = h_small[0];
  DevBuf<uint32_t> d_out;
  II2_TRY(d_out.alloc_scratch(total, s));
  if (total) {
    const unsigned gx = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(1024, (total / np + 2047) / 2048));
    for (uint32_t y0 = 0; y0 < np; y0 += 32768) {
      const uint32_t ny = std::min<uint32_t>(32768, np - y0);
      k_prefix_place<<<dim3(gx, ny), 256, 0, s>>>(recs.p + y0, d_off.p + y0, d_out.p);
      II2_LAUNCHED();
    }
  }
  out->values = own->alloc<uint32_t>(total);
  if (!out->values) return II2_ERR_NOMEM;
  if (total) II2_CUDA_TRY(cudaMemcpyAsync(out->values, d_out.p, total * 4, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaMemcpyAsync(out->value_off, d_off.p, row * 8, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaMemcpyAsync(out->matched, d_mout.p, np, cudaMemcpyDeviceToHost, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  out->_owner = own.release();
  return II2_OK;
}

// ---- in-process gathers (one process, several bound devices) ---------------------------------
int read_gather_devices_impl(const ii2_result* const* parts, int nparts, int root_device,
                             ii2_result** out, cudaStream_t s) {
  GatherArgs b;
  b.world = nparts;
  b.T[0] = b.TB[0] = b.P[0] = 0;
  for (int r = 0; r < nparts; r++) {  // exact counts (a small read's arrays are larger)
    b.T[r + 1] = b.T[r] + parts[r]->T;
    b.TB[r + 1] = b.TB[r] + parts[r]->TB;
    b.P[r + 1] = b.P[r] + parts[r]->P;
  }
  if (b.TB[nparts] >= (1ull << 32) || b.T[nparts] >= 0xFFFFFFFFull) {
    set_last_error("gathered read exceeds 4 GiB of term bytes / 2^32-2 terms");
    return II2_ERR_UNSUPPORTED;
  }
  std::unique_ptr<ii2_result> res(new ii2_result());
  res->stream = s;
  res->has_dec = true;
  res->T = b.T[nparts];
  res->TB = b.TB[nparts];
  res->P = b.P[nparts];
  EmitOut& o = res->out;
  II2_TRY(o.term_bytes.alloc(res->TB, s, 32));
  II2_TRY(o.term_off.alloc(res->T + 1, s, 16));
  II2_TRY(o.post.alloc(res->P, s, 16));
  II2_TRY(o.post_off.alloc(res->T + 1, s, 16));
  // the parts may still be in flight on the streams that produced them
  cudaStream_t waited[kMaxWorld];
  int nwaited = 0;
  for (int r = 0; r < nparts; r++) {
    const ii2_result* p = parts[r];
    cudaStream_t ps = p->stream;
    if (!ps || (ps == s && p->device == root_device)) continue;
    bool seen = false;
    for (int i = 0; i < nwaited && !seen; i++) seen = waited[i] == ps;
    if (seen) continue;
    II2_TRY(stream_wait(s, ps, p->device));
    waited[nwaited++] = ps;
  }
  b.tb = o.term_bytes.p;
  b.toff = o.term_off.p;
  b.post = o.post.p;
  b.poff = o.post_off.p;
  for (int r = 0; r < nparts; r++) {
    const EmitOut& l = parts[r]->out;
    b.src[r] = {l.term_bytes.p, l.term_off.p, l.post.p, l.post_off.p};
  }
  II2_TRY(launch_gather_parts(b, s));
  II2_CUDA_TRY(cudaStreamSynchronize(s));
  *out = res.release();
  return II2_OK;
}

int prefix_gather_devices_impl(const ii2_prefix_out* parts, int nparts, ii2_prefix_out* out,
                               cudaStream_t s) {
  const uint32_t np = nparts ? (uint32_t)parts[0].n_prefixes : 0;
  if (np == 0) return prefix_out_empty(np, out);
  const size_t row = (size_t)np + 1;
  std::vector<uint64_t> vbase(nparts + 1, 0);
  for (int r = 0; r < nparts; r++) vbase[r + 1] = vbase[r] + parts[r].value_off[np];
  // the parts' pinned outputs straight to the root device
  DevBuf<uint64_t> d_voff;
  DevBuf<uint32_t> d_vals;
  DevBuf<uint8_t> d_m;
  II2_TRY(d_voff.alloc_scratch(row * nparts, s));
  II2_TRY(d_vals.alloc_scratch(vbase[nparts], s));
  II2_TRY(d_m.alloc_scratch((size_t)np * nparts, s));
  for (int r = 0; r < nparts; r++) {
    const ii2_prefix_out& p = parts[r];
    II2_CUDA_TRY(cudaMemcpyAsync(d_voff.p + row * r, p.value_off, row * 8, cudaMemcpyHostToDevice, s));
    II2_CUDA_TRY(cudaMemcpyAsync(d_m.p + (size_t)np * r, p.matched, np, cudaMemcpyHostToDevice, s));
    const uint64_t cnt = vbase[r + 1] - vbase[r];
    if (cnt) II2_CUDA_TRY(cudaMemcpyAsync(d_vals.p + vbase[r], p.values, cnt * 4, cudaMemcpyHostToDevice, s));
  }
  return prefix_union_on_root(d_voff.p, d_vals.p, d_m.p, vbase, np, nparts, out, s);
}

}  // namespace

extern "C" {

int ii2_comm_unique_id(uint8_t* id) {
  if (!id) return II2_ERR_INVALID;
  if (!nccl().ok) {
    set_last_error("libnccl.so.2 could not be loaded");
    return II2_ERR_UNSUPPORTED;
  }
  static_assert(sizeof(ncclUniqueId) <= II2_COMM_ID_BYTES, "unique id fits the C-ABI buffer");
  ncclUniqueId u;
  II2_NCCL_TRY(nccl().GetUniqueId(&u));
  memset(id, 0, II2_COMM_ID_BYTES);
  memcpy(id, &u, sizeof(u));
  return II2_OK;
}

int ii2_comm_init(const uint8_t* id, int rank, int world) {
  if (!id || world < 1 || world > kMaxWorld || rank < 0 || rank >= world) return II2_ERR_INVALID;
  II2_TRY(ctx_require());
  if (ctx_device_count() > 1) {
    set_last_error("ii2_comm_init: this process drives several devices (use the in-process gathers)");
    return II2_ERR_INVALID;
  }
  if (!nccl().ok) {
    set_last_error("libnccl.so.2 could not be loaded");
    return II2_ERR_UNSUPPORTED;
  }
  std::lock_guard<std::mutex> lock(g_comm_mu);
  if (g_comm.comm) {
    set_last_error("ii2_comm_init called twice (ii2_comm_shutdown first)");
    return II2_ERR_INVALID;
  }
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  ncclComm_t c = nullptr;
  II2_NCCL_TRY(nccl().CommInitRank(&c, world, u, rank));
  g_comm.comm = c;
  g_comm.rank = rank;
  g_comm.world = world;
  return II2_OK;
}

int ii2_comm_info(int* rank, int* world) {
  if (rank) *rank = g_comm.comm ? g_comm.rank : 0;
  if (world) *world = g_comm.comm ? g_comm.world : 0;
  return II2_OK;
}

void ii2_comm_shutdown(void) {
  std::lock_guard<std::mutex> lock(g_comm_mu);
  if (g_comm.comm) {
    nccl().CommDestroy(g_comm.comm);
    g_comm = Comm();
  }
}

int ii2_read_gather(const ii2_result* local, int root, ii2_result** gathered) {
  if (!local || !gathered) return II2_ERR_INVALID;
  *gathered = nullptr;
  II2_TRY(ctx_require());
  II2_TRY(comm_ready());
  if (root >= g_comm.world || !local->has_dec) return II2_ERR_INVALID;
  cudaStream_t s = cur_stream();
  const int rc = read_gather_impl(local, root, gathered, s);
  if (rc != II2_OK) cudaStreamSynchronize(s);
  arena_reset(s);
  return rc;
}

int ii2_prefix_gather(const ii2_prefix_out* local, int root, ii2_prefix_out* merged) {
  if (!local || !merged) return II2_ERR_INVALID;
  memset(merged, 0, sizeof(*merged));
  II2_TRY(ctx_require());
  II2_TRY(comm_ready());
  if (root >= g_comm.world || (local->n_prefixes && (!local->value_off || !local->matched)))
    return II2_ERR_INVALID;
  cudaStream_t s = cur_stream();
  const int rc = prefix_gather_impl(local, root, merged, s);
  if (rc != II2_OK) {
    cudaStreamSynchronize(s);
    memset(merged, 0, sizeof(*merged));
  }
  arena_reset(s);
  return rc;
}

static int no_device() {
  set_last_error("ii2_init has not succeeded: no CUDA device bound (there is no CPU fallback)");
  return II2_ERR_NO_DEVICE;
}

int ii2_read_gather_devices(const ii2_result* const* parts, int nparts, int root_device,
                            ii2_result** gathered) {
  if (!ctx_ready()) return no_device();
  if (!gathered || nparts < 0 || (nparts && !parts)) return II2_ERR_INVALID;
  *gathered = nullptr;
  if (!ctx_bound(root_device)) {
    set_last_error("root device %d is not in the set bound by ii2_init", root_device);
    return II2_ERR_INVALID;
  }
  if (nparts > kMaxWorld) {
    set_last_error("%d parts in one gather (max %d)", nparts, kMaxWorld);
    return II2_ERR_UNSUPPORTED;
  }
  for (int r = 0; r < nparts; r++) {
    const ii2_result* p = parts[r];
    if (!p || !p->has_dec || !p->out.term_off.p || !p->out.post_off.p) {
      set_last_error("part %d is not a decoded read result", r);
      return II2_ERR_INVALID;
    }
    if (!ctx_peer(root_device, p->device)) {
      set_last_error("part %d lives on device %d, which device %d cannot read (no peer access)", r,
                     p->device, root_device);
      return II2_ERR_UNSUPPORTED;
    }
  }
  II2_TRY(ctx_require_device(root_device));
  cudaStream_t s = cur_stream();
  const int rc = read_gather_devices_impl(parts, nparts, root_device, gathered, s);
  if (rc != II2_OK) cudaStreamSynchronize(s);
  return rc;
}

int ii2_prefix_gather_devices(const ii2_prefix_out* parts, int nparts, int root_device,
                              ii2_prefix_out* merged) {
  if (!ctx_ready()) return no_device();
  if (!merged || nparts < 0 || (nparts && !parts)) return II2_ERR_INVALID;
  memset(merged, 0, sizeof(*merged));
  if (!ctx_bound(root_device)) {
    set_last_error("root device %d is not in the set bound by ii2_init", root_device);
    return II2_ERR_INVALID;
  }
  if (nparts > kMaxWorld) {
    set_last_error("%d parts in one gather (max %d)", nparts, kMaxWorld);
    return II2_ERR_UNSUPPORTED;
  }
  for (int r = 0; r < nparts; r++) {
    const ii2_prefix_out& p = parts[r];
    if (p.n_prefixes != parts[0].n_prefixes) {
      set_last_error("part %d has %llu prefixes, part 0 has %llu", r, (unsigned long long)p.n_prefixes,
                     (unsigned long long)parts[0].n_prefixes);
      return II2_ERR_INVALID;
    }
    if (p.n_prefixes >= 0xFFFFFFFFull) return II2_ERR_INVALID;
    if (p.n_prefixes && (!p.value_off || !p.matched)) return II2_ERR_INVALID;
    if (p.n_prefixes && p.value_off[p.n_prefixes] > 0 && !p.values) {
      set_last_error("part %d holds values but its value array is NULL", r);
      return II2_ERR_INVALID;
    }
  }
  II2_TRY(ctx_require_device(root_device));
  cudaStream_t s = cur_stream();
  const int rc = prefix_gather_devices_impl(parts, nparts, merged, s);
  if (rc != II2_OK) {
    cudaStreamSynchronize(s);
    memset(merged, 0, sizeof(*merged));
  }
  arena_reset(s);
  return rc;
}

}  // extern "C"
