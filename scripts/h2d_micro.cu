// Microbenchmark: how fast can pinned host memory reach HBM on this box?
//   (a) one large cudaMemcpyAsync            (copy engine, the reference point)
//   (b) SM loads of 16 B per lane             (what k_gather_host does)
//   (c) TMA bulk copies host -> shared -> global, a ring of stages per CTA, one thread issues
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -cudart shared -o scripts/h2d_micro scripts/h2d_micro.cu
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1); } } while (0)

__global__ void __launch_bounds__(256) k_ldg(const uint4* __restrict__ src, uint4* __restrict__ dst, uint64_t nvec) {
  const uint64_t tile = 256ull * 4;
  for (uint64_t v0 = (uint64_t)blockIdx.x * tile; v0 < nvec; v0 += (uint64_t)gridDim.x * tile) {
    uint4 x[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const uint64_t v = v0 + u * 256 + threadIdx.x;
      if (v < nvec) x[u] = src[v];
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const uint64_t v = v0 + u * 256 + threadIdx.x;
      if (v < nvec) dst[v] = x[u];
    }
  }
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One thread per CTA drives a ring of STAGES buffers of CHUNK bytes.
template <int STAGES>
__global__ void __launch_bounds__(32) k_tma(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst,
                                            uint64_t bytes, uint32_t chunk) {
  extern __shared__ __align__(128) uint8_t ring[];
  __shared__ __align__(8) uint64_t bar[STAGES];
  if (threadIdx.x != 0) return;
  for (int s = 0; s < STAGES; s++)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[s])));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  const uint64_t nchunk = (bytes + chunk - 1) / chunk;
  // chunks of this CTA: blockIdx.x, + gridDim.x, ...
  uint64_t issued = 0, stored = 0;
  const uint64_t mine = nchunk > blockIdx.x ? (nchunk - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  while (stored < mine) {
    // keep the ring full
    while (issued < mine && issued < stored + STAGES) {
      const int s = (int)(issued % STAGES);
      if (issued >= STAGES) {
        // the store that last read this stage must have finished reading shared memory
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      }
      const uint64_t c = blockIdx.x + issued * gridDim.x;
      const uint64_t at = c * chunk;
      const uint32_t n = (uint32_t)((bytes - at) < chunk ? (bytes - at) : chunk);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bar[s])), "r"(n) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
                       "r"(smem_u32(ring + (size_t)s * chunk)), "l"(src + at), "r"(n), "r"(smem_u32(&bar[s]))
                   : "memory");
      issued++;
    }
    {
      const int s = (int)(stored % STAGES);
      const uint32_t parity = (uint32_t)((stored / STAGES) & 1);
      uint32_t ok = 0;
      while (!ok) {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(ok) : "r"(smem_u32(&bar[s])), "r"(parity) : "memory");
      }
      const uint64_t c = blockIdx.x + stored * gridDim.x;
      const uint64_t at = c * chunk;
      const uint32_t n = (uint32_t)((bytes - at) < chunk ? (bytes - at) : chunk);
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + at),
                   "r"(smem_u32(ring + (size_t)s * chunk)), "r"(n) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      stored++;
    }
  }
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

int main() {
  const uint64_t bytes = 512ull << 20;
  uint8_t *h, *d;
  CK(cudaHostAlloc(&h, bytes, cudaHostAllocDefault));
  CK(cudaMalloc(&d, bytes));
  for (uint64_t i = 0; i < bytes; i += 4) *(uint32_t*)(h + i) = (uint32_t)(i * 2654435761u);
  cudaStream_t s, s2;
  CK(cudaStreamCreate(&s));
  CK(cudaStreamCreate(&s2));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  std::vector<uint8_t> back(bytes);
  auto check = [&](const char* what) {
    CK(cudaMemcpy(back.data(), d, bytes, cudaMemcpyDeviceToHost));
    uint64_t bad = 0;
    for (uint64_t i = 0; i < bytes; i += 4096) bad += back[i] != h[i];
    for (uint64_t i = bytes - 70000; i < bytes; i++) bad += back[i] != h[i];
    if (bad) printf("  !! %s: %llu mismatches\n", what, (unsigned long long)bad);
    CK(cudaMemset(d, 0, bytes));
  };
  auto timeit = [&](const char* what, auto fn) {
    fn();
    CK(cudaStreamSynchronize(s));
    float best = 1e9f;
    for (int r = 0; r < 3; r++) {
      CK(cudaEventRecord(e0, s));
      fn();
      CK(cudaEventRecord(e1, s));
      CK(cudaEventSynchronize(e1));
      float ms;
      CK(cudaEventElapsedTime(&ms, e0, e1));
      if (ms < best) best = ms;
    }
    printf("%-44s %7.2f ms  %6.1f GB/s\n", what, best, bytes / best / 1e6);
    fflush(stdout);
    check(what);
  };
  timeit("cudaMemcpyAsync 512 MB", [&] { CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s)); });
  for (uint64_t piece : {256ull << 10, 1ull << 20, 4ull << 20}) {
    char nm[64];
    snprintf(nm, sizeof nm, "cudaMemcpyAsync pieces of %llu KB", (unsigned long long)(piece >> 10));
    timeit(nm, [&] {
      for (uint64_t at = 0; at < bytes; at += piece) CK(cudaMemcpyAsync(d + at, h + at, piece, cudaMemcpyHostToDevice, s));
    });
  }
  const uint8_t* hd;
  CK(cudaHostGetDevicePointer((void**)&hd, h, 0));
  for (int grid : {16, 32, 64, 148, 296, 592}) {
    char nm[64];
    snprintf(nm, sizeof nm, "ldg.128 kernel, %d CTAs x 256", grid);
    timeit(nm, [&] { k_ldg<<<grid, 256, 0, s>>>((const uint4*)hd, (uint4*)d, bytes / 16); });
  }
  // does the phase of the source matter?  (slices of host arrays start anywhere)
  for (int off : {16, 32, 64, 112}) {
    char nm[64];
    snprintf(nm, sizeof nm, "ldg.128 kernel, 64 CTAs, source phase +%d B", off);
    timeit(nm, [&] { k_ldg<<<64, 256, 0, s>>>((const uint4*)(hd + off), (uint4*)(d + off), bytes / 16 - 8); });
  }
  CK(cudaFuncSetAttribute(k_tma<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 << 10));
  CK(cudaFuncSetAttribute(k_tma<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 << 10));
  for (uint32_t chunk : {2048u, 4096u, 8192u, 16384u, 32768u}) {
    for (int grid : {16, 64, 148, 296}) {
      char nm[64];
      snprintf(nm, sizeof nm, "tma ring 4 x %u B, %d CTAs", chunk, grid);
      timeit(nm, [&] { k_tma<4><<<grid, 32, 4 * chunk, s>>>(hd, d, bytes, chunk); });
    }
  }
  for (uint32_t chunk : {4096u, 16384u}) {
    char nm[64];
    snprintf(nm, sizeof nm, "tma ring 8 x %u B, 64 CTAs", chunk);
    timeit(nm, [&] { k_tma<8><<<64, 32, 8 * chunk, s>>>(hd, d, bytes, chunk); });
  }
  // both at once: copy engine on s2 for the first half, ldg kernel for the second half
  timeit("half copy engine + half ldg kernel", [&] {
    CK(cudaEventRecord(e1, s));
    CK(cudaStreamWaitEvent(s2, e1, 0));
    CK(cudaMemcpyAsync(d, h, bytes / 2, cudaMemcpyHostToDevice, s2));
    k_ldg<<<64, 256, 0, s>>>((const uint4*)(hd + bytes / 2), (uint4*)(d + bytes / 2), bytes / 32);
    cudaEvent_t j;
    CK(cudaEventCreateWithFlags(&j, cudaEventDisableTiming));
    CK(cudaEventRecord(j, s2));
    CK(cudaStreamWaitEvent(s, j, 0));
    CK(cudaEventDestroy(j));
  });
  // both directions at once: is the link full duplex for this traffic?
  uint8_t *h2, *d2;
  CK(cudaHostAlloc(&h2, bytes, cudaHostAllocDefault));
  CK(cudaMalloc(&d2, bytes));
  CK(cudaMemset(d2, 1, bytes));
  auto join_s2 = [&] {
    cudaEvent_t j;
    CK(cudaEventCreateWithFlags(&j, cudaEventDisableTiming));
    CK(cudaEventRecord(j, s2));
    CK(cudaStreamWaitEvent(s, j, 0));
    CK(cudaEventDestroy(j));
  };
  auto fork_s2 = [&] {
    cudaEvent_t j;
    CK(cudaEventCreateWithFlags(&j, cudaEventDisableTiming));
    CK(cudaEventRecord(j, s));
    CK(cudaStreamWaitEvent(s2, j, 0));
    CK(cudaEventDestroy(j));
  };
  timeit("D2H copy engine alone 512 MB", [&] { CK(cudaMemcpyAsync(h2, d2, bytes, cudaMemcpyDeviceToHost, s)); });
  timeit("H2D copy engine + D2H copy engine (512 MB each)", [&] {
    fork_s2();
    CK(cudaMemcpyAsync(h2, d2, bytes, cudaMemcpyDeviceToHost, s2));
    CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s));
    join_s2();
  });
  timeit("H2D ldg kernel + D2H copy engine (512 MB each)", [&] {
    fork_s2();
    CK(cudaMemcpyAsync(h2, d2, bytes, cudaMemcpyDeviceToHost, s2));
    k_ldg<<<64, 256, 0, s>>>((const uint4*)hd, (uint4*)d, bytes / 16);
    join_s2();
  });
  timeit("H2D ldg kernel + D2H copy engine (128 MB)", [&] {
    fork_s2();
    CK(cudaMemcpyAsync(h2, d2, bytes / 4, cudaMemcpyDeviceToHost, s2));
    k_ldg<<<64, 256, 0, s>>>((const uint4*)hd, (uint4*)d, bytes / 16);
    join_s2();
  });
  uint8_t* h2d;
  CK(cudaHostGetDevicePointer((void**)&h2d, h2, 0));
  timeit("D2H stg kernel alone (512 MB), 64 CTAs", [&] {
    k_ldg<<<64, 256, 0, s>>>((const uint4*)d2, (uint4*)h2d, bytes / 16);
  });
  timeit("H2D ldg kernel + D2H stg kernel (512 MB each), 64+64 CTAs", [&] {
    fork_s2();
    k_ldg<<<64, 256, 0, s2>>>((const uint4*)d2, (uint4*)h2d, bytes / 16);
    k_ldg<<<64, 256, 0, s>>>((const uint4*)hd, (uint4*)d, bytes / 16);
    join_s2();
  });
  timeit("H2D ldg kernel + D2H stg kernel (128 MB), 64+64 CTAs", [&] {
    fork_s2();
    k_ldg<<<64, 256, 0, s2>>>((const uint4*)d2, (uint4*)h2d, bytes / 64);
    k_ldg<<<64, 256, 0, s>>>((const uint4*)hd, (uint4*)d, bytes / 16);
    join_s2();
  });
  timeit("H2D ldg kernel + D2H stg kernel (128 MB), 64+8 CTAs", [&] {
    fork_s2();
    k_ldg<<<8, 256, 0, s2>>>((const uint4*)d2, (uint4*)h2d, bytes / 64);
    k_ldg<<<64, 256, 0, s>>>((const uint4*)hd, (uint4*)d, bytes / 16);
    join_s2();
  });
  timeit("H2D copy engine + D2H copy engine (128 MB)", [&] {
    fork_s2();
    CK(cudaMemcpyAsync(h2, d2, bytes / 4, cudaMemcpyDeviceToHost, s2));
    CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s));
    join_s2();
  });
  return 0;
}
