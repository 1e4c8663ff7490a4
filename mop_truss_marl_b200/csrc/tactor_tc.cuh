// tcgen05 building blocks of the whole-network fused actor kernel (tactor_pipe.cuh).
//
//   * a CTA owns 128 rows (8 environments of 16 nodes / 4 of 32) and all 208 (padded) output columns
//   * X.W on the 5th-gen tensor cores: tcgen05.mma kind::f16, M=128 N=208 K=16 per instruction, fp32 accumulators in TMEM
//   * float32-like accuracy inside the fp16 window by the hi/lo split (three MMAs per k-step into the same accumulator)
//   * the B operand (W) sits in shared memory in the canonical no-swizzle K-major layout (8-row x 16-byte core
//     matrices): W is pre-scaled, pre-split and pre-laid-out on the host so a K-chunk is ONE cp.async.bulk (TMA 1-D
//     bulk copy, completion on an mbarrier)
//   * the A operand is generated and split on the fly by the generator threads and written straight into
//     TENSOR MEMORY (tcgen05.st, lane = row, two k per column): it never touches shared memory, whose bandwidth the
//     exchange tiles, the tensor core's B reads, the TMA writes and the epilogue already compete for
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tactor {
namespace tc {

// Operand precision of the split product: x = hi + lo with hi = fp16(x), lo = fp16(x - hi), X.W ~= Xhi.Whi + Xhi.Wlo +
// Xlo.Whi on tcgen05.mma kind::f16 (K = 16 per instruction).  fp16 carries the same 11-bit significand as tf32, so the
// result is float32-like as 3xTF32 is (measured <= 6e-6 on the sigmoid outputs against the float64 oracle) at half
// the operand bytes and twice the tensor rate (3xTF32 on kind::tf32 was the first formulation of this kernel: 0.388 ms
// against 0.382 ms per forward with everything else equal).  What fp16 lacks is range: W is pre-scaled by a power of
// two per layer (undone exactly in the epilogue) and an operand beyond 65504 is reported through tactor_status.  The
// split is float32-like only while the operand is at least 2^-3: below that lo = fp16(x - hi) is an fp16 subnormal, so
// the operand keeps an absolute error of 2^-25 instead of a relative one of 2^-22.  The activations are not scaled by
// the weights' power of two, and a trained actor has most of its mix operands below 2^-3 (DESIGN.md section 3.3): so
// the mix operands X and Y = A.X are carried times a power of two -- XPRE in the five mixes of layer 2 (layer 1's 1/S and
// the pooled Pareto embedding put the factor in), HPRE in the two of layer 3, whose X is the five-way sum H (the layer-2
// epilogues write H times HPRE); the constant bias column of Y carries the factor of its GEMM and the epilogue's 1/S
// takes it out, all exact.  The window of the true activations is [2^-9, 65504 / 64] in layer 2 and [2^-6, 65504 / 8]
// for H, which is larger (a sum of five terms).
constexpr float XPRE = 64.f;
constexpr float HPRE = 8.f;
constexpr int TCM = 128;             // rows per CTA
constexpr int TCN = 208;             // padded output columns (UMMA N, multiple of 16)
constexpr int KCH = 16;              // K elements per chunk (one MMA k-step)
constexpr int KPC = 8;               // K elements per 16-byte core-matrix row
constexpr int NKB = KCH / KPC;       // 16-byte core-matrix columns per chunk
constexpr int SBO = 128;             // bytes between 8-row groups
constexpr int B_LBO = TCN * 16;      // bytes between core matrices adjacent in K (B operand)
constexpr int B_BYTES = NKB * B_LBO; // one of {hi, lo} of a chunk
constexpr int WST = 3;               // W stages in shared memory (K chunks in flight)
constexpr int STAGE_BYTES = 2 * B_BYTES;   // Bhi, Blo of one K chunk
// fp32 accumulate, A and B K-major and f16, M = 128, N = 208
constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(TCN >> 3) << 17) | ((uint32_t)(TCM >> 4) << 24);
constexpr float F16_MAX = 65504.f;
constexpr uint32_t SPIN_LIMIT = 1u << 24;
// W operand image in global memory: per chunk [hi: kb][n][16 bytes = KPC elements] then [lo: ...], STAGE_BYTES in all;
// every chunk is a full K = 16 step (the rows past the bias row k = 200 are zero)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((SBO >> 4) & 0x3FFFu) << 32) | (1ull << 46);        // version 1 (Blackwell), no swizzle
}
// D[tmem] (+)= A[tmem] . B[smem]: A is [128 lanes = rows][8 columns] of tensor memory, two packed fp16 per column, even k
// in the low half (K = 16)
__device__ __forceinline__ void mma_split(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(IDESC), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
               "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
// all MMAs issued so far by this thread have completed -> one arrival on the barrier
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// one lane of the (converged) warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded wait: a mis-programmed barrier must not hang the GPU; returns false on timeout
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t spin = 0; spin < SPIN_LIMIT; ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return true;
  }
  return false;
}
// the same with a pause between polls: a warp that expects to wait long (epilogue between GEMMs, W producer) should not
// keep taking issue slots and mbarrier-unit bandwidth from the warps it waits for
__device__ __forceinline__ bool mbar_wait_relaxed(uint32_t bar, uint32_t parity, uint32_t ns) {
  for (uint32_t spin = 0; spin < SPIN_LIMIT; ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return true;
    if (ns) __nanosleep(ns);
  }
  return false;
}
// the same with acquire semantics at cluster scope
__device__ __forceinline__ bool mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  for (uint32_t spin = 0; spin < SPIN_LIMIT; ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return true;
  }
  return false;
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- warp-level tensor-core pieces of the operand generators (tactor_pipe.cuh) -------------------------------
// D (+)= A.B, m16n8k16, fp16 operands, fp32 accumulators (SASS HMMA.16816.F32).  Fragment ownership (g = lane / 4, t = lane % 4):
//   A [16 x 16] row-major: a0 (row g, k 2t..2t+1)  a1 (row g+8, same k)  a2 (row g, k 2t+8..)  a3 (row g+8, k 2t+8..)
//   B [16 x 8]  col-major: b0 (k 2t..2t+1, col g)  b1 (k 2t+8.., col g)
//   C [16 x 8]           : c0 c1 (row g, cols 2t, 2t+1)  c2 c3 (row g+8, same cols)
__device__ __forceinline__ void hmma16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// three-term split product: c += (ahi + alo).(bhi + blo) without the lo.lo term
// (three independent accumulators joined by FADDs were measured slower: 0.201 against 0.195 ms -- the generators are bound
// by their instruction count, not by the tensor-pipe round trip of the dependent chain)
__device__ __forceinline__ void hmma_split(float* c, const uint32_t* ahi, const uint32_t* alo, const uint32_t* bhi, const uint32_t* blo) {
  hmma16816(c, ahi, bhi[0], bhi[1]);
  hmma16816(c, ahi, blo[0], blo[1]);
  hmma16816(c, alo, bhi[0], bhi[1]);
}
// 16 lanes x 8 columns of tensor memory from the mma accumulator layout: r0 (lane g, column t), r1 (lane g+8, column t),
// r2 (lane g, column 4+t), r3 (lane g+8, column 4+t); the lane field of taddr is the first of the 16 lanes
__device__ __forceinline__ void tmem_st_16x128b_x2(uint32_t taddr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.16x128b.x2.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3])
               : "memory");
}

// counter-based standard normal for the OU noise: element i of tensor `stream_id` (1 = geo, 2 = topo) of call `call`
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ float ou_step(float x, float mu, float theta, float sigma, uint64_t seed, uint64_t call,
                                         uint64_t stream_id, uint64_t i) {
  const uint64_t h = mix64(mix64(seed ^ (call * 0xD1342543DE82EF95ull)) + stream_id * 0x632BE59BD9B4E019ull + i);
  const float u1 = ((uint32_t)(h >> 32) + 1.0f) * 2.3283064365386963e-10f;    // (0, 1]
  const float u2 = (uint32_t)h * 2.3283064365386963e-10f;
  const float nrm = sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
  return x + (theta * (mu - x) * 0.0001f + sigma * nrm);
}

// =========================================================================================================
// Kernel parameters of the whole-network fused actor kernel (tactor_pipe.cuh).
namespace fused {

constexpr int NGEMM = 7;                                   // the seven [200,200] layers: gcn_l2_1..5, gcn_l3_1, gcn_l3_2
constexpr int KH = 200;

struct Params {
  const float* x_n;       // [B,N,13]
  const float* A_n;       // [N,N]
  const float* A_s;       // [B,N,N]
  const float* A_ts;      // [B,N,N]
  const float* A_cs;      // [B,N,N]
  const float* pooled;    // [B,208]
  const float* w1[3];     // layer-1 kernels packed [16,208]
  const float* b1[3];     // [208]
  const float* wimg[NGEMM];
  const float* bias[NGEMM];
  // 1 / (power-of-two scale folded into the fp16 operand images), in DEVICE memory so that a CUDA graph that captured
  // this launch sees the values of the weights it replays with: [0, NGEMM) the seven hidden layers, [NGEMM, NGEMM + 3) the
  // three layer-1 kernels (written by upload_weights next to the images themselves)
  const float* wscale_inv;
  const uint32_t* w1frag;  // [3][13 chunks][32 lanes][8]: mma.sync A fragments (hi a0..a3, lo a0..a3) of [W1k ; b1k]^T, pre-scaled
  const float* w_head[2]; // packed [208,208], first 2 / 3 columns used
  const float* b_head[2];
  float* geo;             // [B,N,2]
  float* topo;            // [B,N,3]
  int M;                  // B*N
  // OU noise of act() (truss2D_RL.py:41-48, 341-350), applied where the sigmoid outputs are written: noise != 0 adds
  // theta*(mu-x)*1e-4 + sigma*n(seed, call, tensor, element); seed_call != nullptr: seed = seed_call[0], call += seed_call[1]
  int noise;
  float mu, theta, sigma;
  uint64_t seed, call;
  const uint64_t* seed_call;
  int n_items;            // work items (full tiles + pieces of split tiles); a persistent CTA walks item, item + grid, ...
  int split_from;         // first work item that is a piece of a tile (tiles of the last partial wave), n_items if none
  int split_f;            // pieces per split tile: 1, 2 or 4
  int* error_flag;
};

}  // namespace fused

}  // namespace tc
}  // namespace tactor
