// Do warp-level mma.sync (HMMA) and tcgen05.mma (UTCHMMA) share the tensor pipe of an SM, and how do they interleave?
// One CTA per SM: warp 0 streams NUTC tcgen05.mma (M=128, N=208, K=16, kind::f16, A from tensor memory, B from shared
// memory, operands are whatever the memories hold), warps 1..NW run NH chained mma.sync.m16n8k16 each.  Prints the cycles of
// each side alone and together.  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -I mop_truss_marl_b200/csrc -o tensor_share scripts/tensor_share.cu
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "tactor_tc.cuh"

using namespace tactor::tc;

__global__ void __launch_bounds__(544, 1) share_kernel(long long* out, int nutc, int nh, int nw, int chain) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&slot)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x == 0) { mbar_init(smem_u32(&bar), 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  for (int i = threadIdx.x; i < 16384 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = slot;
  const long long t0 = clock64();
  long long t1 = t0;
  if (warp == 0) {
    if (nutc > 0) {
      const uint64_t d = make_desc(smem_u32(smem), B_LBO);
      if (elect_one()) {
        for (int i = 0; i < nutc; ++i) mma_split(tmem, tmem + 448, d, i != 0);
        mma_commit(smem_u32(&bar));
      }
      __syncwarp();
      mbar_wait(smem_u32(&bar), 0);
      t1 = clock64();
    }
  } else if (warp <= nw) {
    float c[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) c[i][j] = 0.f;
    const uint32_t a[4] = {0x3c003c00u, 0x3c003c00u, 0x3c003c00u, 0x3c003c00u};
    if (chain == 2) {                                       // no tensor work at all: scale / max / convert (the split sequence's pipes)
      float x[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = (float)(threadIdx.x + i);
      for (int it = 0; it < nh / 4; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = fmaxf(fmaf(x[i], 1.0001f, 0.5f), 1.f);
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(__float_as_uint(x[i]) & 0xffffe000u) + 1e-3f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) c[0][0] += x[i];
    } else if (chain) {
      for (int it = 0; it < nh / 4; ++it)
#pragma unroll
        for (int i = 0; i < 4; ++i) hmma16816(c[0], a, 0x3c003c00u, 0x3c003c00u);     // one dependent chain
    } else {
      for (int it = 0; it < nh / 4; ++it)
#pragma unroll
        for (int i = 0; i < 4; ++i) hmma16816(c[i], a, 0x3c003c00u, 0x3c003c00u);     // four independent chains
    }
    float s = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) s += c[i][0] + c[i][1] + c[i][2] + c[i][3];
    if (s == 12345.678f) out[1000] = (long long)s;
    t1 = clock64();
  }
  if (blockIdx.x == 0 && lane == 0 && warp <= 16) out[warp] = t1 - t0;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
}

// UTC in bursts: `burst` tcgen05.mma back to back, wait for their completion, idle for `gap` cycles, `nburst` times, while
// warps 1..nw run mma.sync continuously until the UTC warp raises a flag; reports how many HMMAs a warp completed.
__global__ void __launch_bounds__(544, 1) burst_kernel(long long* out, int nburst, int burst, int gap, int nw) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  __shared__ volatile int stop;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&slot)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x == 0) { stop = 0; mbar_init(smem_u32(&bar), 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  for (int i = threadIdx.x; i < 16384 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = slot;
  const long long t0 = clock64();
  long long count = 0, busy = 0;
  if (warp == 0) {
    const uint64_t d = make_desc(smem_u32(smem), B_LBO);
    for (int b = 0; b < nburst; ++b) {
      const long long tb = clock64();
      if (elect_one()) {
        for (int i = 0; i < burst; ++i) mma_split(tmem, tmem + 448, d, 1);
        mma_commit(smem_u32(&bar));
      }
      __syncwarp();
      mbar_wait(smem_u32(&bar), b & 1);
      const long long te = clock64();
      busy += te - tb;
      while (clock64() - te < gap) { }
    }
    if (lane == 0) stop = 1;
    count = busy;
  } else if (warp <= nw) {
    float c[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) c[i][j] = 0.f;
    const uint32_t a[4] = {0x3c003c00u, 0x3c003c00u, 0x3c003c00u, 0x3c003c00u};
    while (!stop) {
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int i = 0; i < 4; ++i) hmma16816(c[i], a, 0x3c003c00u, 0x3c003c00u);
      count += 16;
    }
    float s = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) s += c[i][0] + c[i][1] + c[i][2] + c[i][3];
    if (s == 12345.678f) out[1000] = (long long)s;
  }
  const long long t1 = clock64();
  if (blockIdx.x == 0 && lane == 0 && warp <= 16) { out[warp] = t1 - t0; out[32 + warp] = count; }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
}

int main() {
  long long* d;
  cudaMalloc(&d, 8192 * 8);
  cudaFuncSetAttribute(share_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768);
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  auto run = [&](int nutc, int nh, int nw, int chain) {
    long long h[17];
    for (int r = 0; r < 2; ++r) {
      cudaMemset(d, 0, 17 * 8);
      share_kernel<<<sms, 544, 32768>>>(d, nutc, nh, nw, chain);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("{\"error\": \"%s\"}\n", cudaGetErrorString(e)); return; }
    }
    cudaMemcpy(h, d, 17 * 8, cudaMemcpyDeviceToHost);
    long long hm = 0;
    for (int w = 1; w <= nw; ++w) hm = h[w] > hm ? h[w] : hm;
    printf("{\"utc_mmas\": %d, \"hmma_per_warp\": %d, \"hmma_warps\": %d, \"chained\": %d, \"utc_cycles\": %lld, \"utc_cycles_per_mma\": %.1f, "
           "\"hmma_cycles\": %lld, \"hmma_cycles_per_hmma_per_scheduler\": %.2f}\n",
           nutc, nh, nw, chain, h[0], nutc ? (double)h[0] / nutc : 0.0, hm, (nh && nw) ? (double)hm / ((double)nh * ((nw + 3) / 4)) : 0.0);
  };
  run(3000, 0, 0, 0);
  for (int nw : {4, 8, 16}) {                                 // ALU-only warps next to the tcgen05 stream
    run(0, 8192, nw, 2);
    run(3000, 8192, nw, 2);
    run(3000, 32768, nw, 2);
  }
  for (int chain = 0; chain < 2; ++chain)
    for (int nw : {4, 8, 16}) {
      run(0, 8192, nw, chain);
      run(3000, 8192, nw, chain);
      run(3000, 32768, nw, chain);
    }
  cudaFuncSetAttribute(burst_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768);
  auto runb = [&](int nburst, int burst, int gap, int nw) {
    long long h[64];
    for (int r = 0; r < 2; ++r) {
      cudaMemset(d, 0, 64 * 8);
      burst_kernel<<<sms, 544, 32768>>>(d, nburst, burst, gap, nw);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("{\"error\": \"%s\"}\n", cudaGetErrorString(e)); return; }
    }
    cudaMemcpy(h, d, 64 * 8, cudaMemcpyDeviceToHost);
    const double total = (double)h[0], utc_busy = (double)h[32], hm = (double)h[33];
    // HMMA cycles per scheduler = hm * ceil(nw/4) * 8.1 at the uncontended rate
    printf("{\"bursts\": %d, \"mmas_per_burst\": %d, \"gap_cycles\": %d, \"hmma_warps\": %d, \"total_cycles\": %.0f, \"utc_busy_frac\": %.3f, "
           "\"utc_cycles_per_mma\": %.1f, \"hmma_per_warp\": %.0f, \"hmma_pipe_frac_of_idle\": %.3f}\n",
           nburst, burst, gap, nw, total, utc_busy / total, utc_busy / ((double)nburst * burst), hm,
           hm * ((nw + 3) / 4) * 8.1 / (total - utc_busy));
  };
  for (int nw : {8, 16})
    for (int burst : {1, 3, 6, 12})
      for (int gap : {0, 100, 200, 400, 800}) runb(1200 / burst, burst, gap * burst, nw);
  cudaFree(d);
  return 0;
}
