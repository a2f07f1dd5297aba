// Micro-benchmark behind the N-half pipelining decision of tc_exact.cu (run on a B200 through gpurun):
// does the split-fp16 MMA triple (A_hi B_hi -> D1, A_hi B_lo -> D2, A_lo B_hi -> D2), with BOTH operands in shared
// memory (the "ss" form), keep its rate when a K = 256 layer is issued as two N = 128 halves instead of one N = 256
// pass, and with the epilogue's st.shared traffic and the weight ring's bulk copies running beside it?
//   mode 0: N = 256, 16 k-steps x 3 MMAs per layer            (what tc_exact_kernel issues today)
//   mode 1: N = 128, 2 halves x 16 k-steps x 3 MMAs per layer (N-half pipelining)
//   +2: eight warps keep writing 16-byte chunks into the A images (the epilogue's operand stores)
//   +4: one warp keeps pulling 32 KB stages from global memory into a 3-slot ring (the weight stream)
// Build:  nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -I optimalmodulationds_b200/csrc \
//              tools/tcx_ss_microbench.cu -o tools/tcx_ss_microbench
#include <cstdio>
#include <cuda_runtime.h>

#include "tc_ptx.cuh"

using namespace tcx;

constexpr int NT = 12 * 32;
constexpr int OFF_A_HI = 0, OFF_A_LO = 65536, OFF_RING_ = 131072, OFF_BAR_ = OFF_RING_ + 3 * 32768;
constexpr int SMEM = OFF_BAR_ + 128;

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NT, 1)
ss_kernel(int mode, int layers, const uint8_t* gsrc, long long* out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar_done = sbase + OFF_BAR_, bar_ring = sbase + OFF_BAR_ + 8;   // ring barriers: 3 x 8 bytes
  volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(smem + OFF_BAR_ + 64);
  volatile int* stop = reinterpret_cast<volatile int*>(smem + OFF_BAR_ + 96);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  for (int i = tid; i < OFF_BAR_ / 4; i += NT) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u;   // fp16 1.0
  if (tid == 0) *stop = 0;
  if (warp == 8) {
    if (lane == 0) {
      mbar_init(bar_done, 1);
      for (int s = 0; s < 3; ++s) mbar_init(bar_ring + 8 * s, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc_512_2cta(smem_u32((const void*)tmem_ptr));
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  cluster_sync_all();

  if (warp < 8 && (mode & 2)) {
    // epilogue-like stores: every thread rewrites its row's 16-byte chunks of both A images, 32 chunks per image
    uint32_t v = tid;
    uint8_t* a_hi = smem + OFF_A_HI + ((warp & 3) * 32 + lane) * 16;
    uint8_t* a_lo = smem + OFF_A_LO + ((warp & 3) * 32 + lane) * 16;
    while (!*stop) {
#pragma unroll 4
      for (int ch = 0; ch < 16; ++ch) {
        const int c = 16 * (warp >> 2) + ch;
        // ~80 ALU instructions per chunk pair like the real epilogue, so the store RATE is realistic
#pragma unroll
        for (int k = 0; k < 80; ++k) v = v * 1664525u + 1013904223u;
        const uint32_t h = 0x3c003c00u | (v & 0x00010001u);
        *reinterpret_cast<uint4*>(a_hi + c * 2048) = make_uint4(h, h, h, h);
        *reinterpret_cast<uint4*>(a_lo + c * 2048) = make_uint4(h, h, h, h);
      }
    }
  } else if (warp == 9 && (mode & 4)) {
    uint32_t n = 0;
    long long next = clock64();
    while (!*stop) {
      const uint32_t slot = n % 3, use = n / 3;
      if (lane == 0) {
        while (clock64() < next) {}            // the real stream is consumed at 32 KB per 1536 MMA cycles
        next += 1536;
        if (use > 0) mbar_wait(bar_ring + 8 * slot, (use - 1) & 1);
        mbar_expect_tx(bar_ring + 8 * slot, 32768);
        bulk_g2s(sbase + OFF_RING_ + slot * 32768, gsrc + (size_t)((n * 2 + rank) % 52) * 32768, 32768, bar_ring + 8 * slot);
      }
      __syncwarp();
      ++n;
    }
    // drain: wait for the last copies so no bulk copy is in flight at exit
    if (lane == 0)
      for (uint32_t k = (n >= 3 ? n - 3 : 0); k < n; ++k) mbar_wait(bar_ring + 8 * (k % 3), (k / 3) & 1);
  } else if (warp == 8 && rank == 0) {
    const bool half = mode & 1;
    const uint32_t idesc = half ? make_idesc(0, 256, 128) : make_idesc(0, 256, 256);
    const uint32_t b_lbo = half ? 64 * 16 : 128 * 16;
    const uint32_t a_hi = sbase + OFF_A_HI, a_lo = sbase + OFF_A_LO;
    long long c0 = 0, c1 = 0;
    if (elect_one()) {
      c0 = clock64();
      for (int L = 0; L < layers; ++L) {
        for (int x = 0; x < (half ? 2 : 1); ++x)
          for (int st = 0; st < 4; ++st) {
            const uint32_t slot = (uint32_t)(L * 4 + st + 2 * x) % 3;
            const uint32_t b_hi = sbase + OFF_RING_ + slot * 32768, b_lo = b_hi + 16384;
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t ka = (uint32_t)(st * 4 + ks) * 2 * 2048, kb = (uint32_t)ks * 2 * b_lbo;
              const uint64_t adh = make_desc(a_hi + ka, 2048), adl = make_desc(a_lo + ka, 2048);
              const uint64_t bdh = make_desc(b_hi + kb, b_lbo), bdl = make_desc(b_lo + kb, b_lbo);
              const uint32_t acc = (st == 0 && ks == 0) ? 0u : 1u;
              const uint32_t d = tmem_base + (half ? 128u * x : 0u);
              mma_ss_2cta(d, adh, bdh, idesc, acc);
              mma_ss_2cta(d + 256, adh, bdl, idesc, acc);
              mma_ss_2cta(d + 256, adl, bdh, idesc, 1u);
            }
          }
      }
      mma_commit_2cta(bar_done);
      mbar_wait(bar_done, 0);
      c1 = clock64();
      if (blockIdx.x == 0) out[0] = c1 - c0;
      *stop = 1;
    }
    __syncwarp();
  }
  if (warp == 8 && rank == 1) {
    if (lane == 0) mbar_wait(bar_done, 0);
    __syncwarp();
    *stop = 1;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) {
    __syncwarp();
    tmem_free_512_2cta(tmem_base);
  }
}

int main() {
  cudaFuncSetAttribute(ss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
  long long* out;
  cudaMallocManaged(&out, 64);
  uint8_t* g;
  cudaMalloc(&g, 52 * 32768);
  cudaMemset(g, 0, 52 * 32768);
  const int layers = 200;
  const char* names[8] = {"N=256", "N=128 x2", "N=256 +stores", "N=128 x2 +stores", "N=256 +ring", "N=128 x2 +ring",
                          "N=256 +stores +ring", "N=128 x2 +stores +ring"};
  for (int rep = 0; rep < 2; ++rep)
    for (int mode = 0; mode < 8; ++mode) {
      out[0] = 0;
      ss_kernel<<<148, NT, SMEM>>>(mode, layers, g, out);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("mode %d: %s\n", mode, cudaGetErrorString(e)); return 1; }
      printf("%-26s %8.1f cycles / layer (K=256, N=256, 48 MMA-equivalents; floor 6144)\n", names[mode],
             (double)out[0] / layers);
    }
  return 0;
}
