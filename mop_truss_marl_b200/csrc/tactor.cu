// Batched GCN actor forward (include/tactor.h): the 13 GCNConv layers of multimodes_actor
// (train/code/truss2D_RL.py:49-127) for B environments x N nodes at once, plus the OU noise of act().
//
// Two launches per forward:
//   pareto_kernel        Pareto-front branch (gcn_l1_4 + GlobalSumPool) -> pooled [B,208]
//   actor_pipe_kernel    everything else, one CTA per 128 rows, tcgen05 tensor cores (tactor_pipe.cuh)
// (the OU noise of tactor_act is applied by the actor kernel where it writes its outputs).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <new>
#include <string>
#include <vector>

#include "../../include/tactor.h"
#include "../../include/tfem.h"
#include "tactor_tc.cuh"
#include "tactor_pipe.cuh"

namespace tactor {

constexpr int HID = TACTOR_HIDDEN;   // 200
constexpr int LD = 208;              // padded leading dimension of every activation / weight matrix
constexpr int KC = 16;               // layer-1 / head kernels are stored with K padded to a multiple of 16

// ---------------------------------------------------------------------------------------------------------
// Pareto branch (truss2D_RL.py:86-88): x14 = relu(A_p (x_p W14) + b14), summed over the valid Pareto rows
// (GlobalSumPool).  One CTA per environment.
// One CTA per environment: T = x_p W14 [P,200] once, then U = A_p T as a register-tiled product -- thread (p-slice of 13
// rows, 4 feature columns) keeps 13 x 4 accumulators, reads one float4 of T and 13 broadcast entries of A_p per q -- and
// pooled[h] = sum over the valid rows of relu(U[p][h] + b[h]).
constexpr int PSL = 13;                   // Pareto rows per thread slice (4 slices cover P <= 52)
template <int NODES>
__global__ void __launch_bounds__(256)
pareto_kernel(const float* __restrict__ x_p, const float* __restrict__ A_p, const int32_t* __restrict__ n_pf,
              int P, const float* __restrict__ W14, const float* __restrict__ b14, float* __restrict__ pooled_out,
              int B, const int* __restrict__ only_flagged) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (only_flagged) {                      // second pass behind pareto_tri_kernel: only the environments it could not take
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (blockIdx.x < B && only_flagged[blockIdx.x] == 0) return;
  }
  extern __shared__ __align__(16) float psm[];
  float* ts = psm;                        // [P][LD]   x_p W14          (the launch sizes the buffer for this P: a
  float* red = ts + P * LD;               // [4][LD]   per-slice sums     small front keeps many CTAs per SM)
  float* as = red + 4 * LD;               // [P][P]
  float* xs = as + P * P;                 // [P][4]
  const int b = blockIdx.x, tid = threadIdx.x;
  if (b >= B) return;
  for (int i = tid; i < P * 4; i += blockDim.x) xs[i] = x_p[(size_t)b * P * 4 + i];
  for (int i = tid; i < P * P; i += blockDim.x) as[i] = A_p[(size_t)b * P * P + i];
  __syncthreads();
  for (int idx = tid; idx < P * (LD / 4); idx += blockDim.x) {
    const int q = idx / (LD / 4), h4 = idx % (LD / 4);
    const float4 w0 = __ldg(reinterpret_cast<const float4*>(W14 + 0 * LD) + h4), w1 = __ldg(reinterpret_cast<const float4*>(W14 + 1 * LD) + h4);
    const float4 w2 = __ldg(reinterpret_cast<const float4*>(W14 + 2 * LD) + h4), w3 = __ldg(reinterpret_cast<const float4*>(W14 + 3 * LD) + h4);
    const float x0 = xs[q * 4], x1 = xs[q * 4 + 1], x2 = xs[q * 4 + 2], x3 = xs[q * 4 + 3];
    float4 t;                             // same operation order as the scalar form: fma(x3,w3, fma(x2,w2, fma(x1,w1, x0*w0)))
    t.x = fmaf(x3, w3.x, fmaf(x2, w2.x, fmaf(x1, w1.x, x0 * w0.x)));
    t.y = fmaf(x3, w3.y, fmaf(x2, w2.y, fmaf(x1, w1.y, x0 * w0.y)));
    t.z = fmaf(x3, w3.z, fmaf(x2, w2.z, fmaf(x1, w1.z, x0 * w0.z)));
    t.w = fmaf(x3, w3.w, fmaf(x2, w2.w, fmaf(x1, w1.w, x0 * w0.w)));
    reinterpret_cast<float4*>(ts + q * LD)[h4] = t;
  }
  __syncthreads();
  const int valid = n_pf ? min(max(n_pf[b], 0), P) : P;
  const int ps = tid >> 6, h4 = tid & 63;                    // slice = two warps; lanes 52..63 of a slice idle
  if (h4 < LD / 4) {
    float4 acc[PSL];
#pragma unroll
    for (int i = 0; i < PSL; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int p0 = ps * PSL;
    for (int q = 0; q < P; ++q) {
      const float4 t = reinterpret_cast<const float4*>(ts + q * LD)[h4];
#pragma unroll
      for (int i = 0; i < PSL; ++i) {
        if (p0 + i < valid) {                                // warp-uniform
          const float a = as[(p0 + i) * P + q];
          acc[i].x = fmaf(a, t.x, acc[i].x); acc[i].y = fmaf(a, t.y, acc[i].y);
          acc[i].z = fmaf(a, t.z, acc[i].z); acc[i].w = fmaf(a, t.w, acc[i].w);
        }
      }
    }
    const float4 bias = __ldg(reinterpret_cast<const float4*>(b14) + h4);
    float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < PSL; ++i) {
      if (p0 + i < valid) {
        sum.x += fmaxf(acc[i].x + bias.x, 0.f); sum.y += fmaxf(acc[i].y + bias.y, 0.f);
        sum.z += fmaxf(acc[i].z + bias.z, 0.f); sum.w += fmaxf(acc[i].w + bias.w, 0.f);
      }
    }
    reinterpret_cast<float4*>(red + ps * LD)[h4] = sum;
  }
  __syncthreads();
  // the reference's stack-and-reshape scramble (x14b[b,n,h] = pooled[b,(n*200+h)/N]) is applied by the fused
  // kernel's operand generator, so only the pooled embedding is materialised
  if (tid < LD) pooled_out[(size_t)b * LD + tid] = (tid < HID) ? ((red[tid] + red[LD + tid]) + (red[2 * LD + tid] + red[3 * LD + tid])) : 0.f;
}
// Small fronts (P <= PSMALL; the reset-time graph has P = 1): one thread per feature column, everything recomputed in
// registers -- no barrier-separated stages, a few registers, many CTAs per SM (the tiled kernel above needs 3 barriers and
// ~80 registers, which costs more than it saves until the P^2 product dominates).
constexpr int PSMALL = 16;
template <int NODES>
__global__ void __launch_bounds__(256)
pareto_small_kernel(const float* __restrict__ x_p, const float* __restrict__ A_p, const int32_t* __restrict__ n_pf,
                    int P, const float* __restrict__ W14, const float* __restrict__ b14, float* __restrict__ pooled_out,
                    int B, const int* __restrict__ only_flagged) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (only_flagged) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (blockIdx.x < B && only_flagged[blockIdx.x] == 0) return;
  }
  __shared__ float xs[PSMALL * 4];
  __shared__ float as[PSMALL * PSMALL];
  const int b = blockIdx.x, tid = threadIdx.x;
  if (b >= B) return;
  if (tid < P * 4) xs[tid] = x_p[(size_t)b * P * 4 + tid];
  if (tid < P * P) as[tid] = A_p[(size_t)b * P * P + tid];
  __syncthreads();
  const int valid = n_pf ? min(max(n_pf[b], 0), P) : P;
  float sum = 0.f;
  if (tid < HID) {
    const float w0 = W14[0 * LD + tid], w1 = W14[1 * LD + tid], w2 = W14[2 * LD + tid], w3 = W14[3 * LD + tid];
    const float bias = b14[tid];
    if (P == 1) {                         // the reset-time graph (truss2D_ENV.py:348-351): one row, one entry
      const float t0 = fmaf(xs[3], w3, fmaf(xs[2], w2, fmaf(xs[1], w1, xs[0] * w0)));
      if (valid > 0) sum = fmaxf(fmaf(as[0], t0, 0.f) + bias, 0.f);
    } else {
      float t[PSMALL];
#pragma unroll
      for (int q = 0; q < PSMALL; ++q)
        t[q] = (q < P) ? fmaf(xs[q * 4 + 3], w3, fmaf(xs[q * 4 + 2], w2, fmaf(xs[q * 4 + 1], w1, xs[q * 4] * w0))) : 0.f;
      for (int p = 0; p < valid; ++p) {
        float u = 0.f;
#pragma unroll
        for (int q = 0; q < PSMALL; ++q)
          if (q < P) u = fmaf(as[p * P + q], t[q], u);
        sum += fmaxf(u + bias, 0.f);
      }
    }
  }
  if (tid < LD) pooled_out[(size_t)b * LD + tid] = (tid < HID) ? sum : 0.f;
}

// P == 1 (the reset-time graph, truss2D_ENV.py:348-351): pooled[h] = relu(A_p x_p W14[:,h] + b[h]) is five FMAs per
// (environment, column); eight environments per CTA keep the launch from being all CTA-scheduling overhead
constexpr int P1_ENVS = 8;
__global__ void __launch_bounds__(256)
pareto_p1_kernel(const float* __restrict__ x_p, const float* __restrict__ A_p, const int32_t* __restrict__ n_pf,
                 const float* __restrict__ W14, const float* __restrict__ b14, float* __restrict__ pooled_out, int B) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the actor kernel may set itself up beside this one
  const int tid = threadIdx.x;
  if (tid >= LD) return;
  float w0 = 0.f, w1 = 0.f, w2 = 0.f, w3 = 0.f, bias = 0.f;
  if (tid < HID) { w0 = W14[0 * LD + tid]; w1 = W14[1 * LD + tid]; w2 = W14[2 * LD + tid]; w3 = W14[3 * LD + tid]; bias = b14[tid]; }
#pragma unroll
  for (int i = 0; i < P1_ENVS; ++i) {
    const int b = blockIdx.x * P1_ENVS + i;
    if (b >= B) break;
    const float4 x = __ldg(reinterpret_cast<const float4*>(x_p) + b);
    const float a = __ldg(A_p + b);
    const int valid = n_pf ? min(max(n_pf[b], 0), 1) : 1;
    const float t0 = fmaf(x.w, w3, fmaf(x.z, w2, fmaf(x.y, w1, x.x * w0)));   // same operation order as the general kernels
    float sum = 0.f;
    if (valid > 0) sum = fmaxf(fmaf(a, t0, 0.f) + bias, 0.f);
    pooled_out[(size_t)b * LD + tid] = (tid < HID) ? sum : 0.f;
  }
}

// Tridiagonal A_p -- the only Pareto graph the reference builds (pareto_state_data: a chain over the front with self loops,
// symmetrically normalised, zero rows / columns as padding; truss2D_ENV.py:22-41, master_DDPG_truss2D_MO.py:499-517).
// U[p] = a[p][p-1] T[p-1] + a[p][p] T[p] + a[p][p+1] T[p+1] instead of the dense P x P product: one WARP per environment, a
// lane owns the feature columns lane, lane + 32, ..., T slides through three registers per column.  The whole of A_p is still
// read (once, coalesced): an entry outside the band sends the environment to the dense kernel (flag[b] = 1), so any A_p
// gives the same result as before.  Same operation order as the dense kernels (the skipped terms are exact zeros), same
// grouping of the pooled sum, hence bit-identical pooled rows.
constexpr int TRI_WARPS = 8;
__global__ void __launch_bounds__(TRI_WARPS * 32)
pareto_tri_kernel(const float* __restrict__ x_p, const float* __restrict__ A_p, const int32_t* __restrict__ n_pf,
                  int P, const float* __restrict__ W14, const float* __restrict__ b14, float* __restrict__ pooled_out,
                  int B, int* __restrict__ flag) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  __shared__ float diag_s[TRI_WARPS][3][52];
  __shared__ float4 x_s[TRI_WARPS][52];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * TRI_WARPS + warp;
  if (b >= B) return;
  float (*dg)[52] = diag_s[warp];
  // ---- A_p: the three diagonals into shared memory, anything else must be zero ----
  const float* A = A_p + (size_t)b * P * P;
  bool off = false;
  for (int i = lane; i < 3 * 52; i += 32) (&dg[0][0])[i] = 0.f;
  __syncwarp();
  auto take = [&](float v, int i, int j) {
    const int dj = j - i;
    if (dj >= -1 && dj <= 1) dg[dj + 1][i] = v;
    else off = off || (v != 0.f);
  };
  const int PP = P * P;
  if ((PP & 3) == 0 && (reinterpret_cast<uintptr_t>(A) & 15u) == 0) {
    // 128-bit loads, four in flight per lane (the matrix is 10 KB for P = 50: the scan is a latency chain otherwise)
    const float4* A4 = reinterpret_cast<const float4*>(A);
    const int n4 = PP >> 2;
    for (int q0 = lane; q0 < n4; q0 += 128) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int q = q0 + 32 * u;
        v[u] = q < n4 ? __ldg(A4 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int q = q0 + 32 * u;
        if (q < n4) {
          int i = (4 * q) / P, j = 4 * q - i * P;
          const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            take(e[t], i, j);
            if (++j == P) { j = 0; ++i; }
          }
        }
      }
    }
  } else {
    int i = 0, j = lane;
    while (j >= P) { j -= P; ++i; }
    for (int idx = lane; idx < PP; idx += 32) {
      take(__ldg(A + idx), i, j);
      j += 32;
      while (j >= P) { j -= P; ++i; }
    }
  }
  for (int p = lane; p < P; p += 32) x_s[warp][p] = __ldg(reinterpret_cast<const float4*>(x_p + (size_t)b * P * 4) + p);
  off = __any_sync(0xffffffffu, off);
  if (lane == 0) flag[b] = off ? 1 : 0;
  if (off) return;                                           // the dense kernel behind this one takes it
  __syncwarp();
  const int valid = n_pf ? min(max(n_pf[b], 0), P) : P;
  constexpr int NC = 7;                                      // columns per lane: lane + 32 k < 200
  float w0[NC], w1[NC], w2[NC], w3[NC], bias[NC];
#pragma unroll
  for (int k = 0; k < NC; ++k) {
    const int h = lane + 32 * k;
    const bool in = h < HID;
    w0[k] = in ? W14[0 * LD + h] : 0.f; w1[k] = in ? W14[1 * LD + h] : 0.f;
    w2[k] = in ? W14[2 * LD + h] : 0.f; w3[k] = in ? W14[3 * LD + h] : 0.f;
    bias[k] = in ? b14[h] : 0.f;
  }
  auto trow = [&](int p, float* t) {                         // T[p][h] = x_p[p] . W14[:, h], the kernels' common operation order
    const float4 x = (p >= 0 && p < P) ? x_s[warp][p] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < NC; ++k) t[k] = fmaf(x.w, w3[k], fmaf(x.z, w2[k], fmaf(x.y, w1[k], x.x * w0[k])));
  };
  float tp[NC], tc[NC], tn[NC], sum[4][NC];
#pragma unroll
  for (int k = 0; k < NC; ++k) { tp[k] = 0.f; sum[0][k] = sum[1][k] = sum[2][k] = sum[3][k] = 0.f; }
  trow(0, tc);
  // the dense kernel for P > 16 pools in four slices of 13 rows, the small one in a single run: same grouping here
  const int slice = (P > PSMALL) ? PSL : 64;
#pragma unroll
  for (int sl = 0; sl < 4; ++sl) {
    float acc[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) acc[k] = 0.f;
    const int p_end = min(valid, (sl + 1) * slice);
    for (int p = sl * slice; p < p_end; ++p) {
      trow(p + 1, tn);
      const float al = dg[0][p], ad = dg[1][p], au = dg[2][p];
#pragma unroll
      for (int k = 0; k < NC; ++k) {
        float u = 0.f;
        if (p > 0) u = fmaf(al, tp[k], u);
        u = fmaf(ad, tc[k], u);
        if (p + 1 < P) u = fmaf(au, tn[k], u);
        acc[k] += fmaxf(u + bias[k], 0.f);
        tp[k] = tc[k]; tc[k] = tn[k];
      }
    }
#pragma unroll
    for (int k = 0; k < NC; ++k) sum[sl][k] = acc[k];
  }
#pragma unroll
  for (int k = 0; k < NC; ++k) {
    const int h = lane + 32 * k;
    if (h < LD) pooled_out[(size_t)b * LD + h] = (h < HID) ? ((sum[0][k] + sum[1][k]) + (sum[2][k] + sum[3][k])) : 0.f;
  }
}

// tactor_selftest_tmem_layout: every warp stores a tagged accumulator-layout fragment with tcgen05.st.16x128b.x2 at lane
// offsets 0 and 16 and reads its 32 lanes back with the row-per-thread shape (tcgen05.ld.32x32b.x8)
__global__ void __launch_bounds__(128) tmem_layout_selftest_kernel(uint32_t* out) {
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(&slot)), "n"(32) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t base = slot;
  for (int mt = 0; mt < 2; ++mt) {
    uint32_t v[4];
    for (int i = 0; i < 4; ++i) v[i] = 0x1000000u | ((uint32_t)warp << 16) | ((uint32_t)mt << 12) | ((uint32_t)lane << 4) | (uint32_t)i;
    tc::tmem_st_16x128b_x2(base + ((uint32_t)(32 * warp + 16 * mt) << 16), v);
  }
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  __syncwarp();
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(base + ((uint32_t)(32 * warp) << 16)));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  for (int i = 0; i < 8; ++i) out[(32 * warp + lane) * 8 + i] = r[i];
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(32) : "memory");
}

// ---------------------------------------------------------------------------------------------------------
// Device-side rebuild of the weight images (tactor_set_weights_device): the same layouts upload_weights builds on the host.
struct PackArgs {
  const float* kernel[TACTOR_NLAYERS];
  const float* bias[TACTOR_NLAYERS];
  float* d_w[TACTOR_NLAYERS];
  float* d_b[TACTOR_NLAYERS];
  __half* d_wimg[TACTOR_NLAYERS];      // layers 4..10
  uint32_t* w1frag;
  float* wscale_inv;                   // [NGEMM + 3]
  float* wmax;                         // [TACTOR_NLAYERS] scratch: max(|W|, |b|) per layer
};
__constant__ int kInDev[TACTOR_NLAYERS] = {13, 13, 13, 4, 200, 200, 200, 200, 200, 200, 200, 200, 200};
__constant__ int kOutDev[TACTOR_NLAYERS] = {200, 200, 200, 200, 200, 200, 200, 200, 200, 200, 200, 2, 3};

// largest 2^s with wmax 2^s < 2^14 (clamped to 2^+-24), like pow2_scale on the host
__device__ __forceinline__ float pow2_scale_dev(float wmax) {
  int ex = 0;
  if (wmax > 0.f) { frexpf(wmax, &ex); ex = 14 - ex; }
  ex = ex > 24 ? 24 : (ex < -24 ? -24 : ex);
  return ldexpf(1.f, ex);
}

__global__ void __launch_bounds__(256) pack_wmax_kernel(PackArgs a) {
  __shared__ float red[8];
  const int l = blockIdx.x, nW = kInDev[l] * kOutDev[l], nB = kOutDev[l];
  float m = 0.f;
  for (int i = threadIdx.x; i < nW; i += 256) m = fmaxf(m, fabsf(a.kernel[l][i]));
  for (int i = threadIdx.x; i < nB; i += 256) m = fmaxf(m, fabsf(a.bias[l][i]));
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    a.wmax[l] = m;
    const float inv = 1.f / pow2_scale_dev(m);
    if (l >= 4 && l <= 10) a.wscale_inv[l - 4] = inv;
    if (l < 3) a.wscale_inv[tc::fused::NGEMM + l] = inv;
  }
}

// packed [Kpad, 208] kernels and [208] biases of all 13 layers (grid: layer x blocks)
__global__ void __launch_bounds__(256) pack_plain_kernel(PackArgs a) {
  const int l = blockIdx.y, kin = kInDev[l], kout = kOutDev[l];
  const int kpad = (kin + KC - 1) / KC * KC;
  for (int idx = blockIdx.x * 256 + threadIdx.x; idx < kpad * LD; idx += gridDim.x * 256) {
    const int i = idx / LD, o = idx - i * LD;
    a.d_w[l][idx] = (i < kin && o < kout) ? a.kernel[l][(size_t)i * kout + o] : 0.f;
  }
  if (blockIdx.x == 0 && threadIdx.x < LD) a.d_b[l][threadIdx.x] = threadIdx.x < kout ? a.bias[l][threadIdx.x] : 0.f;
}

// tcgen05 operand images of the seven [200,200] layers (grid: layer 4..10 x blocks): per 16-wide K chunk
// [hi | lo][kb][n][8 halfs]; row k = 200 holds the bias
__global__ void __launch_bounds__(256) pack_img_kernel(PackArgs a) {
  const int l = 4 + blockIdx.y, K = kInDev[l], kout = kOutDev[l];
  const int bn = tc::TCN, kpc = tc::KPC, nkb = tc::KCH / kpc;
  const int nch = (K + 1 + tc::KCH - 1) / tc::KCH;
  const int total = nch * 2 * nkb * bn * kpc;
  const float scale = pow2_scale_dev(a.wmax[l]);
  for (int idx = blockIdx.x * 256 + threadIdx.x; idx < total; idx += gridDim.x * 256) {
    int r = idx;
    const int t = r % kpc; r /= kpc;
    const int n = r % bn; r /= bn;
    const int kb = r % nkb; r /= nkb;
    const int part = r % 2; r /= 2;
    const int c = r;
    const int k = c * tc::KCH + kpc * kb + t;
    float v = 0.f;
    if (n < kout && k < K) v = a.kernel[l][(size_t)k * kout + n] * scale;
    else if (n < kout && k == K) v = a.bias[l][n] * scale;
    const __half hi = __float2half_rn(v);
    a.d_wimg[l][idx] = part == 0 ? hi : __float2half_rn(v - __half2float(hi));
  }
}

// mma.sync A fragments of [W1k ; b1k]^T for the three layer-1 kernels: [3][13 chunks][hi | lo][32 lanes][4]
__global__ void __launch_bounds__(32) pack_w1frag_kernel(PackArgs a) {
  const int l = blockIdx.y, c = blockIdx.x, lane = threadIdx.x, kout = kOutDev[l];
  const float scale = pow2_scale_dev(a.wmax[l]);
  auto we = [&](int cc, int f) -> float {
    if (f >= kout || cc > 13) return 0.f;
    return (cc < 13 ? a.kernel[l][(size_t)cc * kout + f] : a.bias[l][f]) * scale;
  };
  auto pack = [](float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
    const __half l0 = __float2half_rn(x0 - __half2float(h0)), l1 = __float2half_rn(x1 - __half2float(h1));
    hi = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
    lo = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
  };
  const int g = lane / 4, t = lane % 4, f0 = c * tc::KCH + g;
  uint32_t* hi = a.w1frag + (((size_t)l * tc::pipe::NCH + c) * 2 + 0) * 128 + (size_t)lane * 4;
  uint32_t* lo = a.w1frag + (((size_t)l * tc::pipe::NCH + c) * 2 + 1) * 128 + (size_t)lane * 4;
  pack(we(2 * t, f0), we(2 * t + 1, f0), hi[0], lo[0]);
  pack(we(2 * t, f0 + 8), we(2 * t + 1, f0 + 8), hi[1], lo[1]);
  pack(we(2 * t + 8, f0), we(2 * t + 9, f0), hi[2], lo[2]);
  pack(we(2 * t + 8, f0 + 8), we(2 * t + 9, f0 + 8), hi[3], lo[3]);
}

// 12-node graphs (the 6 x 2 shapes of train/code) run on the 16-node build: every environment is padded to 16 rows with zero
// features and zero adjacency rows / columns (a padded node neither sends nor receives), the kernel divides the pooled
// scramble by the real node count and writes only the real rows.
__global__ void __launch_bounds__(256)
pad_nodes_kernel(int B, int n, const float* __restrict__ x_n, const float* __restrict__ A_n, const float* __restrict__ A_s,
                 const float* __restrict__ A_ts, const float* __restrict__ A_cs, float* __restrict__ x_o, float* __restrict__ An_o,
                 float* __restrict__ As_o, float* __restrict__ Ats_o, float* __restrict__ Acs_o) {
  constexpr int NP = 16;
  const int per_env = NP * 13 + 3 * NP * NP;
  const long long total = (long long)B * per_env;
  for (long long idx = (long long)blockIdx.x * 256 + threadIdx.x; idx < total; idx += (long long)gridDim.x * 256) {
    const int b = (int)(idx / per_env), r = (int)(idx % per_env);
    if (r < NP * 13) {
      const int i = r / 13, c = r % 13;
      x_o[(size_t)b * NP * 13 + r] = i < n ? x_n[((size_t)b * n + i) * 13 + c] : 0.f;
    } else {
      const int t = (r - NP * 13) / (NP * NP), e = (r - NP * 13) % (NP * NP), i = e / NP, j = e % NP;
      const float* src = t == 0 ? A_s : t == 1 ? A_ts : A_cs;
      float* dst = t == 0 ? As_o : t == 1 ? Ats_o : Acs_o;
      dst[(size_t)b * NP * NP + e] = (i < n && j < n) ? src[((size_t)b * n + i) * n + j] : 0.f;
    }
  }
  if (blockIdx.x == 0)
    for (int e = threadIdx.x; e < NP * NP; e += 256) {
      const int i = e / NP, j = e % NP;
      An_o[e] = (i < n && j < n) ? A_n[i * n + j] : 0.f;
    }
}

constexpr int pareto_smem(int P) { return (P * LD + 4 * LD + P * P + P * 4) * 4; }
constexpr int PARETO_SMEM = pareto_smem(50);

}  // namespace tactor

// =========================================================================================================
namespace {
thread_local std::string g_actor_err;
}
struct tactor_handle_s {
  int device = 0, nodes = 0, max_batch = 0;
  int n_real = 0;                      // nodes of the caller's graphs (12: padded to 16 internally; else = nodes)
  float* pad[5] = {};                  // padded x_n, A_n, A_s, A_n_ts, A_n_cs of a 12-node handle
  float* d_w[TACTOR_NLAYERS] = {};     // packed [Kpad, 208]
  float* d_b[TACTOR_NLAYERS] = {};     // [208]
  float* pooled = nullptr;             // [max_batch, 208] Pareto embedding
  int* pareto_flag = nullptr;          // [max_batch] 1 = A_p of this environment is not tridiagonal (dense kernel takes it)
  int pareto_dense = 0;                // TACTOR_PARETO_DENSE=1: always the dense kernels (A/B timing, tests)
  float* d_wimg[TACTOR_NLAYERS] = {};  // tcgen05 operand image of the hidden layers (hi/lo split, core-matrix layout)
  uint32_t* d_w1frag = nullptr;        // mma.sync A-fragment image of the three layer-1 kernels (tactor_pipe.cuh)
  float* d_wmax = nullptr;             // [13] scratch of tactor_set_weights_device
  float* d_wscale_inv = nullptr;       // [NGEMM + 3] 1 / power-of-two scale of d_wimg[4 + g] and of the three layer-1 images
  int* d_error = nullptr;              // set by a kernel whose mbarrier wait timed out
  int sms = 0;                         // SM count of the device (persistent grid, tile splitting of the last wave); TACTOR_NO_SPLIT=1:
                                       // one CTA per unsplit tile
  std::atomic<int64_t> launches{0};
  uint64_t calls = 0;
};

namespace {
int afail(int code, const std::string& msg) { g_actor_err = msg; return code; }
const int kIn[TACTOR_NLAYERS] = {13, 13, 13, 4, 200, 200, 200, 200, 200, 200, 200, 200, 200};
const int kOut[TACTOR_NLAYERS] = {200, 200, 200, 200, 200, 200, 200, 200, 200, 200, 200, 2, 3};

struct Guard {
  int prev = -1;
  explicit Guard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); }
  ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};

template <int NODES, int NREAL = NODES>
cudaError_t launch_pipe(tactor::tc::fused::Params& p, int M, int sms, cudaStream_t st) {
  using namespace tactor;
  const int tiles = (M + tc::TCM - 1) / tc::TCM;
  // wave quantisation: one CTA per SM, so `tiles % sms` tiles would run as a last wave that leaves most SMs idle.
  // Cut those tiles into 2 or 4 row pieces (one CTA each) when the pieces still fit one wave.
  int grid = tiles;
  p.split_from = grid; p.split_f = 1;
  if (sms > 0) {
    const int rem = tiles % sms, full = tiles - rem;
    const int f = (rem > 0 && 4 * rem <= sms) ? 4 : (rem > 0 && 2 * rem <= sms) ? 2 : 1;
    if (f > 1) { p.split_from = full; p.split_f = f; grid = full + f * rem; }
  }
  p.n_items = grid;
  if (sms > 0 && grid > sms) grid = sms;                   // persistent: one CTA per SM walks the items
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)tc::pipe::PTHREADS);
  cfg.dynamicSmemBytes = tc::pipe::pipe_smem_bytes<NODES>();
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  // programmatic dependent launch: the kernel's set-up (TMEM, barriers, weights) runs beside the Pareto-branch kernel that
  // precedes it; the generators wait (griddepcontrol.wait) before they touch its output or the state tensors
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 2;
  return cudaLaunchKernelEx(&cfg, tc::pipe::actor_pipe_kernel<NODES, NREAL>, p);
}

template <int NODES, int NREAL = NODES>
cudaError_t set_pipe_smem() {
  return cudaFuncSetAttribute(tactor::tc::pipe::actor_pipe_kernel<NODES, NREAL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              tactor::tc::pipe::pipe_smem_bytes<NODES>());
}

// (re)builds the device copies of the weights: packed [Kpad,208] kernels / [208] biases and the tcgen05 operand
// images of the seven [200,200] layers.  Buffers are allocated on first use and overwritten afterwards.
cudaError_t upload_weights(tactor_handle_s* h, const tactor_weights* w) {
  cudaError_t e = cudaSuccess;
  for (int l = 0; l < TACTOR_NLAYERS && e == cudaSuccess; ++l) {
    const int kin = kIn[l], kout = kOut[l];
    const int kpad = (kin + tactor::KC - 1) / tactor::KC * tactor::KC;
    std::vector<float> wp((size_t)kpad * tactor::LD, 0.f), bp(tactor::LD, 0.f);
    for (int i = 0; i < kin; ++i)
      for (int o = 0; o < kout; ++o) wp[(size_t)i * tactor::LD + o] = w->kernel[l][(size_t)i * kout + o];
    for (int o = 0; o < kout; ++o) bp[o] = w->bias[l][o];
    if (!h->d_w[l]) e = cudaMalloc(&h->d_w[l], wp.size() * 4);
    if (e == cudaSuccess && !h->d_b[l]) e = cudaMalloc(&h->d_b[l], bp.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_w[l], wp.data(), wp.size() * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_b[l], bp.data(), bp.size() * 4, cudaMemcpyHostToDevice);
  }
  // tcgen05 operand images of the [200,200] layers: per 16-wide K chunk, [hi|lo][kb][n][8 halfs].  W is scaled by S = 2^s (largest s with max(|W|, |b|) S < 2^14, so that hi and lo stay
  // normal fp16 numbers), hi = fp16(W S), lo = fp16(W S - hi); the kernel's epilogue multiplies the accumulator by 1/S
  // (exact).  Row k = 200 of the image (inside the zero-padded tail chunk) holds the bias: the generators feed a constant
  // 1 in column 200 of A.
  float wscale_inv[tactor::tc::fused::NGEMM + 3];
  auto pow2_scale = [](float wmax, float& scale, float& inv) {     // largest 2^s with wmax 2^s < 2^14
    int ex = 0;
    if (wmax > 0.f) { frexpf(wmax, &ex); ex = 14 - ex; }            // wmax in [2^(e-1), 2^e): wmax * 2^(14-e) < 2^14
    ex = ex > 24 ? 24 : (ex < -24 ? -24 : ex);
    scale = ldexpf(1.f, ex);
    inv = ldexpf(1.f, -ex);
  };
  for (int l = 4; l <= 10 && e == cudaSuccess; ++l) {
    const int K = kIn[l], kout = kOut[l];
    float wmax = 0.f;
    for (size_t i = 0; i < (size_t)K * kout; ++i) wmax = fmaxf(wmax, fabsf(w->kernel[l][i]));
    for (int i = 0; i < kout; ++i) wmax = fmaxf(wmax, fabsf(w->bias[l][i]));
    if (!(wmax < INFINITY)) return cudaErrorInvalidValue;
    float scale;
    pow2_scale(wmax, scale, wscale_inv[l - 4]);
    std::vector<__half> img;
    const int kpc = tactor::tc::KPC, nkb = tactor::tc::KCH / kpc;
    for (int c = 0; c * tactor::tc::KCH < K + 1; ++c)
      for (int part = 0; part < 2; ++part)
        for (int kb = 0; kb < nkb; ++kb)
          for (int n = 0; n < tactor::tc::TCN; ++n)
            for (int t = 0; t < kpc; ++t) {
              const int k = c * tactor::tc::KCH + kpc * kb + t;
              float v = 0.f;
              if (n < kout && k < K) v = w->kernel[l][(size_t)k * kout + n] * scale;
              else if (n < kout && k == K) v = w->bias[l][n] * scale;         // A's column K is the constant 1
              const __half hi = __float2half_rn(v);
              img.push_back(part == 0 ? hi : __float2half_rn(v - __half2float(hi)));
            }
    if (!h->d_wimg[l]) e = cudaMalloc(&h->d_wimg[l], img.size() * sizeof(__half));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_wimg[l], img.data(), img.size() * sizeof(__half), cudaMemcpyHostToDevice);
  }
  // mma.sync A fragments of [W1k ; b1k]^T (the generators' layer-1 product X^T = relu([W1k ; b1k]^T . [Z, 1]^T)): per
  // layer-1 kernel, per 16-feature chunk, [hi | lo][lane][a0..a3]; lane (g = lane / 4, t = lane % 4) holds
  // a0 (feature g, c 2t..2t+1)  a1 (feature g+8, same c)  a2 (feature g, c 2t+8..)  a3 (feature g+8, c 2t+8..), c = 13 is
  // the bias.  Scaled by a power of two like the hidden layers (the generator multiplies by 1/S, exact).
  std::vector<uint32_t> frag((size_t)tactor::tc::pipe::W1F_WORDS, 0u);
  for (int l = 0; l < 3 && e == cudaSuccess; ++l) {
    const int kout = kOut[l];
    float wmax = 0.f;
    for (size_t i = 0; i < (size_t)13 * kout; ++i) wmax = fmaxf(wmax, fabsf(w->kernel[l][i]));
    for (int i = 0; i < kout; ++i) wmax = fmaxf(wmax, fabsf(w->bias[l][i]));
    if (!(wmax < INFINITY)) return cudaErrorInvalidValue;
    float scale;
    pow2_scale(wmax, scale, wscale_inv[tactor::tc::fused::NGEMM + l]);
    auto we = [&](int c, int f) -> float {
      if (f >= kout || c > 13) return 0.f;
      return (c < 13 ? w->kernel[l][(size_t)c * kout + f] : w->bias[l][f]) * scale;
    };
    auto pack = [](float x0, float x1, uint32_t& hi, uint32_t& lo) {
      const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
      const __half l0 = __float2half_rn(x0 - __half2float(h0)), l1 = __float2half_rn(x1 - __half2float(h1));
      uint16_t b[4];
      memcpy(&b[0], &h0, 2); memcpy(&b[1], &h1, 2); memcpy(&b[2], &l0, 2); memcpy(&b[3], &l1, 2);
      hi = (uint32_t)b[0] | ((uint32_t)b[1] << 16);
      lo = (uint32_t)b[2] | ((uint32_t)b[3] << 16);
    };
    for (int c = 0; c < tactor::tc::pipe::NCH; ++c)
      for (int lane = 0; lane < 32; ++lane) {
        const int g = lane / 4, t = lane % 4, f0 = c * tactor::tc::KCH + g;
        uint32_t* hi = &frag[(((size_t)l * tactor::tc::pipe::NCH + c) * 2 + 0) * 128 + (size_t)lane * 4];
        uint32_t* lo = &frag[(((size_t)l * tactor::tc::pipe::NCH + c) * 2 + 1) * 128 + (size_t)lane * 4];
        pack(we(2 * t, f0), we(2 * t + 1, f0), hi[0], lo[0]);
        pack(we(2 * t, f0 + 8), we(2 * t + 1, f0 + 8), hi[1], lo[1]);
        pack(we(2 * t + 8, f0), we(2 * t + 9, f0), hi[2], lo[2]);
        pack(we(2 * t + 8, f0 + 8), we(2 * t + 9, f0 + 8), hi[3], lo[3]);
      }
  }
  if (e == cudaSuccess && !h->d_w1frag) e = cudaMalloc(&h->d_w1frag, frag.size() * 4);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_w1frag, frag.data(), frag.size() * 4, cudaMemcpyHostToDevice);
  // the scales live in device memory: a CUDA graph that captured a forward of this handle (trollout_step_host) reads the
  // values that belong to the weight images it replays with
  if (e == cudaSuccess && !h->d_wscale_inv) e = cudaMalloc(&h->d_wscale_inv, sizeof(wscale_inv));
  if (e == cudaSuccess) e = cudaMemcpy(h->d_wscale_inv, wscale_inv, sizeof(wscale_inv), cudaMemcpyHostToDevice);
  return e;
}

struct Noise {
  int on = 0;
  float mu = 0.f, theta = 0.f, sigma = 0.f;
  uint64_t seed = 0, call = 0;
  const uint64_t* seed_call = nullptr;
};

template <int NODES>
cudaError_t run_forward(tactor_handle_s* h, int B, const tactor_inputs* in, float* geo, float* topo, const Noise& nz,
                        cudaStream_t st) {
  using namespace tactor;
  const int M = B * NODES;
  float* pooled = h->pooled;
  if (in->P == 1 && (reinterpret_cast<uintptr_t>(in->x_p) & 15u) == 0)
    pareto_p1_kernel<<<(B + P1_ENVS - 1) / P1_ENVS, 256, 0, st>>>(in->x_p, in->A_p, in->n_pf, h->d_w[3], h->d_b[3], pooled, B);
  else {
    // the chain graph of pareto_state_data is tridiagonal: one warp per environment; environments with any entry outside
    // the band are flagged and redone by the dense kernel, which returns at once for the others
    const int* only = nullptr;
    if (!h->pareto_dense && (reinterpret_cast<uintptr_t>(in->x_p) & 15u) == 0) {
      pareto_tri_kernel<<<(B + TRI_WARPS - 1) / TRI_WARPS, TRI_WARPS * 32, 0, st>>>(in->x_p, in->A_p, in->n_pf, in->P, h->d_w[3],
                                                                                   h->d_b[3], pooled, B, h->pareto_flag);
      only = h->pareto_flag;
      h->launches.fetch_add(1);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)B); cfg.blockDim = dim3(256); cfg.stream = st;
    cfg.dynamicSmemBytes = in->P <= PSMALL ? 0 : pareto_smem(in->P);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = only ? 1 : 0;
    if (in->P <= PSMALL)
      cudaLaunchKernelEx(&cfg, pareto_small_kernel<NODES>, in->x_p, in->A_p, in->n_pf, (int)in->P, (const float*)h->d_w[3],
                         (const float*)h->d_b[3], pooled, B, only);
    else
      cudaLaunchKernelEx(&cfg, pareto_kernel<NODES>, in->x_p, in->A_p, in->n_pf, (int)in->P, (const float*)h->d_w[3],
                         (const float*)h->d_b[3], pooled, B, only);
  }
  tc::fused::Params p{};
  p.x_n = in->x_n; p.A_n = in->A_n; p.A_s = in->A_s; p.A_ts = in->A_n_ts; p.A_cs = in->A_n_cs; p.pooled = pooled;
  for (int k = 0; k < 3; ++k) { p.w1[k] = h->d_w[k]; p.b1[k] = h->d_b[k]; }
  for (int g = 0; g < tc::fused::NGEMM; ++g) { p.wimg[g] = h->d_wimg[4 + g]; p.bias[g] = h->d_b[4 + g]; }
  p.wscale_inv = h->d_wscale_inv; p.w1frag = h->d_w1frag;
  p.w_head[0] = h->d_w[11]; p.w_head[1] = h->d_w[12]; p.b_head[0] = h->d_b[11]; p.b_head[1] = h->d_b[12];
  p.geo = geo; p.topo = topo; p.M = M; p.error_flag = h->d_error;
  p.noise = nz.on; p.mu = nz.mu; p.theta = nz.theta; p.sigma = nz.sigma; p.seed = nz.seed; p.call = nz.call; p.seed_call = nz.seed_call;
  cudaError_t e = (h->n_real == 12) ? launch_pipe<16, 12>(p, M, h->sms, st)      // the padded 12-node build
                                    : launch_pipe<NODES>(p, M, h->sms, st);
  h->launches.fetch_add(2);
  return e != cudaSuccess ? e : cudaGetLastError();
}
}  // namespace

extern "C" {

const char* tactor_last_error(void) { return g_actor_err.c_str(); }

int tactor_create(const tactor_weights* w, int nodes, int max_batch, int device, tactor_handle_t* out) {
  if (!w || !out) return afail(TFEM_ERR_ARG, "null argument");
  *out = nullptr;
  if (nodes != 12 && nodes != 16 && nodes != 32) return afail(TFEM_ERR_UNSUPPORTED, "nodes must be 12, 16 or 32");
  const int n_real = nodes;
  if (nodes == 12) nodes = 16;          // 12-node graphs (train/code) are padded to the 16-node build, see pad_nodes_kernel
  if (max_batch <= 0) return afail(TFEM_ERR_ARG, "max_batch must be positive");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return afail(TFEM_ERR_CUDA, "no CUDA device: no CPU path");
  if (device < 0 || device >= ndev) return afail(TFEM_ERR_ARG, "bad device index");
  tactor_handle_s* h = new (std::nothrow) tactor_handle_s();
  if (!h) return afail(TFEM_ERR_ARG, "out of host memory");
  h->device = device; h->nodes = nodes; h->n_real = n_real; h->max_batch = max_batch;
  Guard g(device);
  for (int l = 0; l < TACTOR_NLAYERS; ++l)
    if (!w->kernel[l] || !w->bias[l]) { tactor_destroy(h); return afail(TFEM_ERR_ARG, "missing layer weights"); }
  cudaError_t e = upload_weights(h, w);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, device);
  if (const char* v = getenv("TACTOR_NO_SPLIT")) { if (v[0] == '1') h->sms = 0; }
  if (e == cudaSuccess) e = cudaMalloc(&h->d_error, 65536);
  if (e == cudaSuccess) e = cudaMemset(h->d_error, 0, 65536);
  if (e == cudaSuccess) e = (nodes == 16) ? set_pipe_smem<16>() : set_pipe_smem<32>();
  if (e == cudaSuccess && n_real == 12) e = set_pipe_smem<16, 12>();
  if (e == cudaSuccess)
    e = (nodes == 16) ? cudaFuncSetAttribute(tactor::pareto_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, tactor::PARETO_SMEM)
                      : cudaFuncSetAttribute(tactor::pareto_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, tactor::PARETO_SMEM);
  if (e == cudaSuccess) e = cudaMalloc(&h->pooled, (size_t)max_batch * tactor::LD * 4);
  if (e == cudaSuccess) e = cudaMalloc(&h->pareto_flag, (size_t)max_batch * sizeof(int));
  if (n_real != nodes) {
    const size_t sz[5] = {(size_t)max_batch * 16 * 13, 16 * 16, (size_t)max_batch * 256, (size_t)max_batch * 256, (size_t)max_batch * 256};
    for (int k = 0; k < 5 && e == cudaSuccess; ++k) e = cudaMalloc(&h->pad[k], sz[k] * sizeof(float));
  }
  if (const char* v = getenv("TACTOR_PARETO_DENSE")) h->pareto_dense = (v[0] == '1');
  if (e != cudaSuccess) { tactor_destroy(h); return afail(TFEM_ERR_CUDA, std::string("actor setup: ") + cudaGetErrorString(e)); }
  *out = h;
  return TFEM_OK;
}

int tactor_set_weights(tactor_handle_t h, const tactor_weights* w) {
  if (!h || !w) return afail(TFEM_ERR_ARG, "null argument");
  for (int l = 0; l < TACTOR_NLAYERS; ++l)
    if (!w->kernel[l] || !w->bias[l]) return afail(TFEM_ERR_ARG, "missing layer weights");
  Guard g(h->device);
  cudaError_t e = cudaDeviceSynchronize();                  // no forward of this handle may still read the old weights
  if (e == cudaSuccess) e = upload_weights(h, w);
  if (e != cudaSuccess) return afail(TFEM_ERR_CUDA, std::string("actor weights: ") + cudaGetErrorString(e));
  return TFEM_OK;
}

int tactor_set_weights_device(tactor_handle_t h, const tactor_weights* w, void* stream) {
  if (!h || !w) return afail(TFEM_ERR_ARG, "null argument");
  for (int l = 0; l < TACTOR_NLAYERS; ++l)
    if (!w->kernel[l] || !w->bias[l]) return afail(TFEM_ERR_ARG, "missing layer weights");
  Guard g(h->device);
  cudaError_t e = cudaSuccess;
  if (!h->d_wmax) e = cudaMalloc(&h->d_wmax, TACTOR_NLAYERS * sizeof(float));
  if (e != cudaSuccess) return afail(TFEM_ERR_CUDA, std::string("actor weights: ") + cudaGetErrorString(e));
  tactor::PackArgs a{};
  for (int l = 0; l < TACTOR_NLAYERS; ++l) {
    a.kernel[l] = w->kernel[l]; a.bias[l] = w->bias[l];
    a.d_w[l] = h->d_w[l]; a.d_b[l] = h->d_b[l];
    a.d_wimg[l] = reinterpret_cast<__half*>(h->d_wimg[l]);
  }
  a.w1frag = h->d_w1frag; a.wscale_inv = h->d_wscale_inv; a.wmax = h->d_wmax;
  cudaStream_t st = (cudaStream_t)stream;
  tactor::pack_wmax_kernel<<<TACTOR_NLAYERS, 256, 0, st>>>(a);
  tactor::pack_plain_kernel<<<dim3(16, TACTOR_NLAYERS), 256, 0, st>>>(a);
  tactor::pack_img_kernel<<<dim3(32, 7), 256, 0, st>>>(a);
  tactor::pack_w1frag_kernel<<<dim3(tactor::tc::pipe::NCH, 3), 32, 0, st>>>(a);
  e = cudaGetLastError();
  h->launches.fetch_add(4);
  if (e != cudaSuccess) return afail(TFEM_ERR_CUDA, std::string("actor weights: ") + cudaGetErrorString(e));
  return TFEM_OK;
}

int tactor_destroy(tactor_handle_t h) {
  if (!h) return TFEM_OK;
  Guard g(h->device);
  for (int l = 0; l < TACTOR_NLAYERS; ++l) { if (h->d_w[l]) cudaFree(h->d_w[l]); if (h->d_b[l]) cudaFree(h->d_b[l]); }
  if (h->pooled) cudaFree(h->pooled);
  if (h->pareto_flag) cudaFree(h->pareto_flag);
  for (float* p : h->pad) if (p) cudaFree(p);
  for (int l = 0; l < TACTOR_NLAYERS; ++l) if (h->d_wimg[l]) cudaFree(h->d_wimg[l]);
  if (h->d_error) cudaFree(h->d_error);
  if (h->d_w1frag) cudaFree(h->d_w1frag);
  if (h->d_wscale_inv) cudaFree(h->d_wscale_inv);
  if (h->d_wmax) cudaFree(h->d_wmax);
  delete h;
  return TFEM_OK;
}

static int check_inputs(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo) {
  if (!h || !in || !geo || !topo) return afail(TFEM_ERR_ARG, "null argument");
  if (B < 0 || B > h->max_batch) return afail(TFEM_ERR_ARG, "batch exceeds max_batch");
  if (!in->x_n || !in->A_n || !in->A_s || !in->A_n_ts || !in->A_n_cs || !in->x_p || !in->A_p)
    return afail(TFEM_ERR_ARG, "x_n, A_n, A_s, A_n_ts, A_n_cs, x_p and A_p are required");
  if (in->P < 1 || in->P > 50) return afail(TFEM_ERR_ARG, "P must be in 1..50 (MAX_FRONT)");
  const void* vec[] = {in->A_n, in->A_s, in->A_n_ts, in->A_n_cs, in->x_n};     // read with 128-bit loads / 16-byte async copies
  for (const void* p : vec)
    if (h->n_real == h->nodes && (reinterpret_cast<uintptr_t>(p) & 15u))
      return afail(TFEM_ERR_ALIGN, "x_n and the adjacency tensors must be 16-byte aligned");
  return TFEM_OK;
}

static int forward_impl(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo, const Noise& nz,
                        void* stream) {
  if (int rc = check_inputs(h, B, in, geo, topo)) return rc;
  if (B == 0) return TFEM_OK;
  Guard g(h->device);
  tactor_inputs padded;
  if (h->n_real != h->nodes) {          // 12 -> 16 nodes: zero-padded copies of the graph tensors in handle-owned buffers
    const long long total = (long long)B * (16 * 13 + 3 * 256);
    const int grid = (int)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
    tactor::pad_nodes_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(B, h->n_real, in->x_n, in->A_n, in->A_s, in->A_n_ts, in->A_n_cs,
                                                                      h->pad[0], h->pad[1], h->pad[2], h->pad[3], h->pad[4]);
    h->launches.fetch_add(1);
    padded = *in;
    padded.x_n = h->pad[0]; padded.A_n = h->pad[1]; padded.A_s = h->pad[2]; padded.A_n_ts = h->pad[3]; padded.A_n_cs = h->pad[4];
    in = &padded;
  }
  cudaError_t e = (h->nodes == 16) ? run_forward<16>(h, B, in, geo, topo, nz, (cudaStream_t)stream)
                                   : run_forward<32>(h, B, in, geo, topo, nz, (cudaStream_t)stream);
  if (e != cudaSuccess) return afail(TFEM_ERR_CUDA, std::string("actor forward: ") + cudaGetErrorString(e));
  return TFEM_OK;
}

int tactor_forward(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo, void* stream) {
  return forward_impl(h, B, in, geo, topo, Noise{}, stream);
}

// the OU noise is applied by the actor kernel itself where it writes the sigmoid outputs (no extra launch)
int tactor_act(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo, float mu, float theta,
               float sigma, uint64_t seed, void* stream) {
  Noise nz;
  if (h && B > 0 && !(sigma == 0.f && theta == 0.f)) {
    nz.on = 1; nz.mu = mu; nz.theta = theta; nz.sigma = sigma; nz.seed = seed; nz.call = h->calls;
  }
  const int rc = forward_impl(h, B, in, geo, topo, nz, stream);
  if (rc == TFEM_OK && nz.on) h->calls++;
  return rc;
}

int tactor_act_dev(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo, float mu, float theta,
                   float sigma, const uint64_t* seed_call_dev, uint32_t call_offset, void* stream) {
  if (!seed_call_dev) return afail(TFEM_ERR_ARG, "null argument");
  Noise nz;
  if (B > 0 && !(sigma == 0.f && theta == 0.f)) {
    nz.on = 1; nz.mu = mu; nz.theta = theta; nz.sigma = sigma; nz.call = call_offset; nz.seed_call = seed_call_dev;
  }
  return forward_impl(h, B, in, geo, topo, nz, stream);
}

uint64_t tactor_reserve_calls(tactor_handle_t h, uint32_t n, int64_t replayed_launches) {
  if (!h) return 0;
  const uint64_t base = h->calls;
  h->calls += n;
  h->launches.fetch_add(replayed_launches);
  return base;
}

int64_t tactor_launch_count(tactor_handle_t h) { return h ? h->launches.load() : 0; }

int tactor_selftest_tmem_layout(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return afail(TFEM_ERR_CUDA, "no such CUDA device");
  Guard g(device);
  uint32_t* d = nullptr;
  std::vector<uint32_t> hbuf(128 * 8, 0u);
  cudaError_t e = cudaMalloc(&d, hbuf.size() * 4);
  if (e == cudaSuccess) e = cudaMemset(d, 0, hbuf.size() * 4);
  if (e == cudaSuccess) { tactor::tmem_layout_selftest_kernel<<<1, 128>>>(d); e = cudaGetLastError(); }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(hbuf.data(), d, hbuf.size() * 4, cudaMemcpyDeviceToHost);
  if (d) cudaFree(d);
  if (e != cudaSuccess) return afail(TFEM_ERR_CUDA, std::string("tmem self-test: ") + cudaGetErrorString(e));
  // register i of lane (g = lane / 4, t = lane % 4) of block mt -> TMEM lane 16 mt + g + 8 (i & 1), column t + 4 (i >> 1)
  for (int warp = 0; warp < 4; ++warp)
    for (int mt = 0; mt < 2; ++mt)
      for (int lane = 0; lane < 32; ++lane)
        for (int i = 0; i < 4; ++i) {
          const int row = 32 * warp + 16 * mt + lane / 4 + 8 * (i & 1), col = lane % 4 + 4 * (i >> 1);
          const uint32_t want = 0x1000000u | ((uint32_t)warp << 16) | ((uint32_t)mt << 12) | ((uint32_t)lane << 4) | (uint32_t)i;
          if (hbuf[row * 8 + col] != want) {
            char msg[160];
            snprintf(msg, sizeof msg, "tcgen05.st.16x128b.x2 layout differs: warp %d block %d lane %d reg %d expected at (%d,%d), found 0x%x there",
                     warp, mt, lane, i, row, col, hbuf[row * 8 + col]);
            return afail(TFEM_ERR_UNSUPPORTED, msg);
          }
        }
  return TFEM_OK;
}

int tactor_status(tactor_handle_t h) {
  if (!h) return afail(TFEM_ERR_ARG, "null argument");
  Guard g(h->device);
  int flag = 0;
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(&flag, h->d_error, 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && flag) e = cudaMemset(h->d_error, 0, 4);          // reported once: later forwards are judged on their own
  if (e != cudaSuccess) return afail(TFEM_ERR_CUDA, std::string("actor status: ") + cudaGetErrorString(e));
  if (flag & 1) return afail(TFEM_ERR_CUDA, "an mbarrier wait timed out inside actor_pipe_kernel");
  if (flag & 2) return afail(TFEM_ERR_UNSUPPORTED, "an activation left the fp16 range of the split tensor-core product (|A.X| > 65504 or NaN input)");
  return TFEM_OK;
}

#ifdef TACTOR_PROF
// development build only (python -m mop_truss_marl_b200.build --prof -> lib/libtfem_prof.so, scripts/actor_prof.py): the
// per-warp cycle counters CTA 0 of the last actor_pipe_kernel launch left behind the error flag
int tactor_prof_read(tactor_handle_t h, long long* out, int n) {
  if (!h || !out || n < 0 || n > 8000) return afail(TFEM_ERR_ARG, "bad argument");
  Guard g(h->device);
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(out, h->d_error + 32, (size_t)n * 8, cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? TFEM_OK : afail(TFEM_ERR_CUDA, cudaGetErrorString(e));
}
#endif

}  // extern "C"
