// bench_gather.cu -- ceiling for the emit kernel's memory pattern: out[i] = in[perm[i]] for 80-byte records
// (16-byte pieces, 5 lanes per record, streaming stores), no checksum, no framing.  Prints ms and GB/s moved.
// Variants: LDG.128 into registers, per-thread cp.async (LDGSTS) into shared memory, bulk copies (TMA), cudaMemcpy.
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o tools/bench_gather tools/bench_gather.cu
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

__device__ __forceinline__ uint4 ldg_stream_v4(const void *p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream_v4(void *p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__global__ void k_fill_perm(uint32_t *perm, uint32_t n, uint32_t mul) {
  // a bijection on [0, n) for n = 10^8: i * mul mod n with gcd(mul, n) = 1
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
    perm[i] = (uint32_t)((i * (uint64_t)mul) % n);
}

template <int UNROLL>
__global__ void __launch_bounds__(256) k_gather(const uint8_t *__restrict__ in, const uint32_t *__restrict__ perm,
                                                uint8_t *__restrict__ out, uint64_t npieces) {
  // piece q = 5 * record + c
  const uint64_t stride = (uint64_t)gridDim.x * 256 * UNROLL;
  for (uint64_t base = (uint64_t)blockIdx.x * 256 * UNROLL; base < npieces; base += stride) {
    uint4 v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; u++) {
      uint64_t q = base + threadIdx.x + u * 256;
      if (q < npieces) {
        uint32_t r = (uint32_t)(q / 5), c = (uint32_t)(q - 5ull * r);
        v[u] = ldg_stream_v4(in + (uint64_t)perm[r] * 80 + 16 * c);
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; u++) {
      uint64_t q = base + threadIdx.x + u * 256;
      if (q < npieces) stg_stream_v4(out + q * 16, v[u]);
    }
  }
}

// ---------------------------------------------------------------------------------------------- TMA (bulk async copy) variants
// One bulk copy per 80-byte record: cp.async.bulk.shared::cluster.global lands the record in a 16-byte aligned slot of a
// shared-memory ring and completes on the stage's mbarrier (no register staging, no LSU work for the gather).
// MODE 0: the stage leaves the SM as ONE cp.async.bulk.global.shared::cta of 256 * 80 bytes (data never touches registers).
// MODE 1: consumer warps read the stage with LDS.128 and write it out with streaming STG.128 (what a kernel that must
//         look at the bytes -- checksum -- has to do).
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

constexpr int TILE_RECS = 256;
constexpr int TILE_BYTES = TILE_RECS * 80;

template <int STAGES, int MODE, int PW, int CONSUMER_WARPS>
__global__ void __launch_bounds__(32 * (PW + CONSUMER_WARPS)) k_gather_tma(const uint8_t *__restrict__ in, const uint32_t *__restrict__ perm,
                                                                           uint8_t *__restrict__ out, uint32_t ntiles) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem);  // [STAGES] full, [STAGES] empty
  uint8_t *ring = smem + 256;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + STAGES);
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(full0 + 8 * s, PW);
      mbar_init(empty0 + 8 * s, MODE == 0 ? 1 : CONSUMER_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  constexpr int RPL = 8 / PW;  // records per producer lane and tile
  if (warp < PW) {
    // ---- producers: the issue of a bulk copy is a warp-uniform instruction (UBLKCP): per-lane addresses are serialised
    //      by the compiler (elect / R2UR / branch, ~8 instructions per copy), so several warps share a tile
    uint32_t it = 0;
    uint32_t nxt[RPL];
    uint32_t tile = blockIdx.x;
    const uint32_t r0 = warp * (TILE_RECS / PW) + lane * RPL;
    if (tile < ntiles)
      for (int k = 0; k < RPL; k++) nxt[k] = perm[(uint64_t)tile * TILE_RECS + r0 + k];
    for (; tile < ntiles; tile += gridDim.x, it++) {
      const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
      uint32_t idx[RPL];
      for (int k = 0; k < RPL; k++) idx[k] = nxt[k];
      if (tile + gridDim.x < ntiles)
        for (int k = 0; k < RPL; k++) nxt[k] = perm[(uint64_t)(tile + gridDim.x) * TILE_RECS + r0 + k];
      if (it >= STAGES) mbar_wait(empty0 + 8 * s, ph ^ 1u);
      const uint32_t bar = full0 + 8 * s;
      if (lane == 0) mbar_expect_tx(bar, TILE_BYTES / PW);
      __syncwarp();
      const uint32_t dst = smem_u32(ring + (size_t)s * TILE_BYTES) + r0 * 80;
#pragma unroll
      for (int k = 0; k < RPL; k++) bulk_g2s(dst + k * 80, in + (uint64_t)idx[k] * 80, 80, bar);
    }
  } else {
    // ---- consumers
    const int cw = warp - PW;
    uint32_t it = 0;
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it++) {
      const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
      mbar_wait(full0 + 8 * s, ph);
      uint8_t *dstg = out + (uint64_t)tile * TILE_BYTES;
      if (MODE == 0) {
        if (cw == 0 && lane == 0) {
          bulk_s2g(dstg, smem_u32(ring + (size_t)s * TILE_BYTES), TILE_BYTES);
          bulk_commit();
          bulk_wait_read<0>();
          mbar_arrive(empty0 + 8 * s);
        }
      } else {
        const uint4 *src = reinterpret_cast<const uint4 *>(ring + (size_t)s * TILE_BYTES);
        const int ct = cw * 32 + lane;
#pragma unroll 5
        for (int q = ct; q < TILE_BYTES / 16; q += 32 * CONSUMER_WARPS) stg_stream_v4(dstg + 16 * q, src[q]);
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * s);
      }
    }
  }
}

template <int STAGES, int MODE, int PW, int CW>
static void run_tma(const uint8_t *in, const uint32_t *perm, uint8_t *out, uint32_t n, int ctas_per_sm, cudaEvent_t e0, cudaEvent_t e1) {
  const size_t smem = 256 + (size_t)STAGES * TILE_BYTES;
  cudaFuncSetAttribute(k_gather_tma<STAGES, MODE, PW, CW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const uint32_t ntiles = n / TILE_RECS;
  for (int rep = 0; rep < 2; rep++) {
    cudaEventRecord(e0);
    k_gather_tma<STAGES, MODE, PW, CW><<<148 * ctas_per_sm, 32 * (PW + CW), smem>>>(in, perm, out, ntiles);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep) printf("TMA gather (one 80 B bulk copy per record), %s, %d stages, %d producer + %d consumer warps, %d CTAs/SM: %.3f ms, %.0f GB/s  [%s]\n",
                    MODE == 0 ? "bulk store" : "LDS+STG store", STAGES, PW, CW, ctas_per_sm, ms, (double)n * 164 / (ms * 1e-3) / 1e9,
                    cudaGetErrorString(cudaGetLastError()));
  }
}

// ---------------------------------------------------------------------------------------------- LDGSTS (cp.async) variant
// Per-thread asynchronous copies: each thread lands its 5 pieces of a 256-record tile with cp.async.cg (16 B, SASS
// LDGSTS) in a thread-private ring of D stages (piece u of thread t in stage s at [s][u][t]), one commit group per
// tile, and writes a tile out with LDS.128 + STG.128 once cp.async.wait_group D-1 says it landed.  No barriers: only
// the issuing thread reads a slot.  The CTA's dynamic shared memory is padded to `smem` so that the run has the
// occupancy and L1 carve-out of the emit kernel it models.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint4 lds_v4(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}

template <int D>
__global__ void __launch_bounds__(256) k_gather_ldgsts(const uint8_t *__restrict__ in, const uint32_t *__restrict__ perm,
                                                       uint8_t *__restrict__ out, uint32_t ntiles) {
  extern __shared__ __align__(16) uint8_t smem[];
  const uint32_t ring = smem_u32(smem) + 16u * threadIdx.x;  // + (s * 5 + u) * 4096
  uint32_t tile = blockIdx.x;
  // record indices of the next tile to issue, one tile ahead of the issue
  uint32_t idx[5];
  auto load_idx = [&](uint32_t t) {
#pragma unroll
    for (int u = 0; u < 5; u++) {
      const uint32_t q = u * 256 + threadIdx.x, r = q / 5;
      idx[u] = t < ntiles ? perm[(uint64_t)t * TILE_RECS + r] : 0u;
    }
  };
  auto issue = [&](uint32_t t, int s) {
    if (t < ntiles) {
#pragma unroll
      for (int u = 0; u < 5; u++) {
        const uint32_t q = u * 256 + threadIdx.x, c = q - 5 * (q / 5);
        cp_async16(ring + (s * 5 + u) * 4096u, in + (uint64_t)idx[u] * 80 + 16 * c);
      }
    }
    cp_async_commit();  // empty groups past the end keep the group count per tile uniform
  };
  load_idx(tile);
#pragma unroll
  for (int s = 0; s < D; s++) {
    const uint32_t t = tile + s * gridDim.x;
    issue(t, s);
    load_idx(t + gridDim.x);
  }
  for (int s = 0; tile < ntiles; tile += gridDim.x, s = s + 1 == D ? 0 : s + 1) {
    cp_async_wait<D - 1>();
    uint8_t *dst = out + (uint64_t)tile * TILE_BYTES + 16 * threadIdx.x;
#pragma unroll
    for (int u = 0; u < 5; u++) stg_stream_v4(dst + u * 4096, lds_v4(ring + (s * 5 + u) * 4096u));
    const uint32_t t = tile + D * gridDim.x;
    issue(t, s);
    load_idx(t + gridDim.x);
  }
}

template <int D>
static void run_ldgsts(const uint8_t *in, const uint32_t *perm, uint8_t *out, uint32_t n, int ctas_per_sm, size_t smem,
                       cudaEvent_t e0, cudaEvent_t e1) {
  cudaFuncSetAttribute(k_gather_ldgsts<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gather_ldgsts<D>, 256, smem);
  const uint32_t ntiles = n / TILE_RECS;
  for (int rep = 0; rep < 3; rep++) {
    cudaEventRecord(e0);
    k_gather_ldgsts<D><<<148 * ctas_per_sm, 256, smem>>>(in, perm, out, ntiles);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep) printf("LDGSTS gather (cp.async.cg 16 B, thread-private ring), D = %d, %d CTAs/SM (%d resident), %.1f KB smem/CTA: %.3f ms, %.0f GB/s  [%s]\n",
                    D, ctas_per_sm, per_sm, smem / 1024.0, ms, (double)n * 164 / (ms * 1e-3) / 1e9, cudaGetErrorString(cudaGetLastError()));
  }
}

static void check_copy(const uint8_t *d_in, const uint32_t *d_perm, const uint8_t *d_out, uint32_t n) {
  // spot check: records 0, 1, n/2 of the output equal the permuted input
  uint32_t probe[3] = {0, 1, (n / 256) * 256 - 1};
  for (uint32_t r : probe) {
    uint32_t pr;
    uint8_t a[80], b[80];
    cudaMemcpy(&pr, d_perm + r, 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(a, d_in + (size_t)pr * 80, 80, cudaMemcpyDeviceToHost);
    cudaMemcpy(b, d_out + (size_t)r * 80, 80, cudaMemcpyDeviceToHost);
    bool ok = true;
    for (int i = 0; i < 80; i++) ok &= a[i] == b[i];
    if (!ok) printf("MISMATCH at record %u\n", r);
  }
}

__global__ void k_fill_data(uint32_t *p, uint64_t words) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < words; i += (uint64_t)gridDim.x * blockDim.x)
    p[i] = (uint32_t)(i * 2654435761u) ^ (uint32_t)(i >> 7);
}

int main(int argc, char **argv) {
  const uint32_t n = argc > 1 ? (uint32_t)atoll(argv[1]) : 100000000u;
  uint8_t *in, *out;
  uint32_t *perm;
  cudaMalloc(&in, (size_t)n * 80);
  cudaMalloc(&out, (size_t)n * 80);
  cudaMalloc(&perm, (size_t)n * 4);
  k_fill_data<<<148 * 8, 256>>>(reinterpret_cast<uint32_t *>(in), (uint64_t)n * 20);
  k_fill_perm<<<148 * 8, 256>>>(perm, n, 48271u * 7919u + 2u * 3u * 0u + 0u | 1u);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  const uint64_t npieces = (uint64_t)n * 5;
  for (int ctas : {2, 3, 4, 6, 8}) {
    for (int rep = 0; rep < 2; rep++) {
      cudaEventRecord(e0);
      k_gather<5><<<148 * ctas, 256>>>(in, perm, out, npieces);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms;
      cudaEventElapsedTime(&ms, e0, e1);
      if (rep) printf("gather-copy 80 B records, unroll 5, %d CTAs/SM: %.3f ms, %.0f GB/s (84 B/rec read + 80 B/rec write)\n", ctas, ms,
                      (double)n * 164 / (ms * 1e-3) / 1e9);
    }
  }
  // LDGSTS variants, each at the shared-memory footprint k_emit_fast4 has with that ring (emit_pipe.cuh, Emit4Smem):
  // 5120 B tables + 22016 B image + (D+1) KB indices + BATCH KB partials + 32 B per parked tile + (D+3) * 32 B
  // descriptors + D * 20 KB ring.  Only the (CTAs/SM, D, BATCH) that fit 228 KB per SM (1 KB reserved per CTA).
  auto fe4_smem = [](int d, int batch) { return (size_t)5120 + 22016 + (d + 1) * 1024 + batch * 1024 + batch * 32 + (d + 3) * 32 + d * 20480; };
  cudaMemset(out, 0, (size_t)n * 80);
  run_ldgsts<1>(in, perm, out, n, 2, fe4_smem(1, 8), e0, e1);
  check_copy(in, perm, out, n);
  run_ldgsts<2>(in, perm, out, n, 2, fe4_smem(2, 8), e0, e1);
  run_ldgsts<3>(in, perm, out, n, 2, fe4_smem(3, 8), e0, e1);
  run_ldgsts<1>(in, perm, out, n, 3, fe4_smem(1, 8), e0, e1);
  cudaMemset(out, 0, (size_t)n * 80);
  run_ldgsts<2>(in, perm, out, n, 3, fe4_smem(2, 4), e0, e1);
  check_copy(in, perm, out, n);
  run_ldgsts<1>(in, perm, out, n, 4, fe4_smem(1, 4), e0, e1);
  // TMA variants
  cudaMemset(out, 0, (size_t)n * 80);
  run_tma<4, 0, 1, 1>(in, perm, out, n, 2, e0, e1);
  check_copy(in, perm, out, n);
  run_tma<4, 0, 2, 1>(in, perm, out, n, 2, e0, e1);
  run_tma<4, 0, 4, 1>(in, perm, out, n, 2, e0, e1);
  run_tma<8, 0, 4, 1>(in, perm, out, n, 1, e0, e1);
  run_tma<8, 0, 8, 1>(in, perm, out, n, 1, e0, e1);
  run_tma<3, 0, 4, 1>(in, perm, out, n, 3, e0, e1);
  run_tma<2, 0, 4, 1>(in, perm, out, n, 4, e0, e1);
  run_tma<2, 0, 2, 1>(in, perm, out, n, 4, e0, e1);
  cudaMemset(out, 0, (size_t)n * 80);
  run_tma<4, 1, 4, 4>(in, perm, out, n, 2, e0, e1);
  check_copy(in, perm, out, n);
  run_tma<4, 1, 2, 6>(in, perm, out, n, 2, e0, e1);
  run_tma<3, 1, 2, 6>(in, perm, out, n, 3, e0, e1);
  run_tma<3, 1, 4, 4>(in, perm, out, n, 3, e0, e1);
  run_tma<8, 1, 8, 8>(in, perm, out, n, 1, e0, e1);
  // sequential copy of the same volume for reference
  for (int rep = 0; rep < 2; rep++) {
    cudaEventRecord(e0);
    cudaMemcpyAsync(out, in, (size_t)n * 80, cudaMemcpyDeviceToDevice);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep) printf("cudaMemcpy D2D %.3f ms, %.0f GB/s\n", ms, (double)n * 160 / (ms * 1e-3) / 1e9);
  }
  printf("%s\n", cudaGetErrorString(cudaGetLastError()));
  return 0;
}
