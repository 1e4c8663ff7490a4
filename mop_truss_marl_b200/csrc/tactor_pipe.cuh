// Whole-network fused actor kernel, fully pipelined ("pipe") formulation.
//
// One CTA carries a 128-row tile (ENVS environments of NODES nodes) through all 13
// GCNConv layers of multimodes_actor.call (train/code/truss2D_RL.py:75-127).  The adjacency product is moved IN FRONT
// of the dense contraction,
//
//      A_g . (X_g . W_g) + b_g   ==   [A_g . X_g, 1] . [W_g ; b_g]        (spektral GCNConv, associativity)
//
// so that the tensor-core epilogue is row-local (scale, ReLU, accumulate) and four groups of warps run concurrently,
// coupled only by mbarriers:
//
//   generators  warps 0..4 NPH-1   row group q = warp & 3 (the warp's 32 rows = 2 environments of 16 nodes / 1 of 32),
//                            chunk phase ph = warp >> 2: the warp owns every NPH-th 16-wide K chunk.  EVERYTHING it does
//                            is a chain of warp-level tensor-core products (mma.sync m16n8k16, fp16 hi/lo split, fp32
//                            accumulators) whose accumulator fragments are re-used as the next product's operand
//                            fragments, so nothing is exchanged through shared memory:
//                              Z    = A_n . x_n                      once per item   (gcn_l1_1..3 share it)
//                              X^T  = relu([W1k ; b1k]^T . [Z, 1]^T) per chunk       (layer 1, features x rows)
//                              Y    = A_g . X                        per chunk       (the C fragment of X^T IS the B
//                                                                                     fragment of this product)
//                            then Y = hi + lo in fp16 -> tcgen05.st.16x128b straight from the accumulator layout into the
//                            A stage (TMEM, two k per column).  gcn_l2_5 takes X from the pooled Pareto embedding (the
//                            reference's reshape scramble), layer 3 from H (shared memory).  The stage is acquired right
//                            before the store and published in the middle of the warp's next chunk (hand_off).
//   producer    1 warp       streams the pre-split W chunks into shared memory (cp.async.bulk, mbarrier tx),
//                            running ahead across GEMM boundaries
//   issuer      1 warp       tcgen05.mma kind::f16 (Yhi.Whi + Yhi.Wlo + Ylo.Whi), A from tensor memory, B from
//                            shared memory, accumulator g&1 of two (TMEM columns [0,208) and [256,464))
//   epilogue    NEPIW warps  tcgen05.ld the finished accumulator while the next GEMM is already running (one warp per
//                            32-row group): relu(D / S) -> H (+)= (g <= 4), or the sigmoid heads gcn_l4_1/2 (g = 5, 6);
//                            the bias is row 200 of the W image (A's column 200 is the constant XPRE or HPRE, tactor_tc.cuh)
//
// TMEM map (512 columns): [0,208) acc0 | [208,256) A stages hi (6 x 8 columns of packed pairs) | [256,464) acc1
//                         | [464,512) A stages lo
#pragma once
#include <cuda_fp16.h>

#include <type_traits>

#include "tactor_tc.cuh"

namespace tactor {
namespace tc {
namespace pipe {

using fused::Params;
using fused::NGEMM;
using fused::KH;

constexpr int PAST = 6;                                     // A-operand stages in tensor memory
constexpr int ACOLS = 8;                                    // TMEM columns of one A stage (two fp16 k per 32-bit column)
constexpr int MAXST = 6;                                    // barrier slots per ring
constexpr int TM_ACC1 = 256, TM_AHI = 208, TM_ALO = 464;
constexpr int LDH = 204;                                    // padded row length of the H tile (2 LDH = 24 mod 32: the B-fragment
                                                            // loads of layer 3 -- 4 row pairs x 8 features -- hit 32 distinct banks)
constexpr int NCH = (KH + KCH - 1) / KCH;                   // 13 chunks per GEMM
constexpr int W1F_WORDS = 3 * NCH * 2 * 32 * 4;             // layer-1 fragment image: [3][13][hi | lo][32 lanes][4]
// warp roles: 4 NPH generators, NEPIW epilogue warps, issuer, W producer.  Measured fastest for both node counts against
// 1, 3 or 4 generator phases and 8 epilogue warps (profiles/README.md)
constexpr int NPH = 2;                                      // generator phases: a generator warp owns every NPH-th chunk
constexpr int NEPIW = 4;                                    // epilogue warps, one per 32-row group
constexpr int PTHREADS = (4 * NPH + NEPIW + 2) * 32;

template <int NODES>
__host__ __device__ constexpr int pipe_smem_bytes() {
  return WST * STAGE_BYTES + TCM * LDH * 4 + W1F_WORDS * 4 + 2 * (TCM / NODES) * 208 * 4 + 2 * TCM * 13 * 4 +
         2 * NODES * NODES * 4 + 2 * 201 * 4 * 4 + 2 * TCM * 4 * 4 + 384;
}

__device__ __forceinline__ uint32_t h2_bits(const __half2& h) { return *reinterpret_cast<const uint32_t*>(&h); }
// (x0, x1) = hi + lo in fp16, x0 in the low half
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 f = __half22float2(h);
  hi = h2_bits(h);
  lo = h2_bits(__floats2half2_rn(x0 - f.x, x1 - f.y));
}
// tcgen05.ld of 8 accumulator columns without the wait (software pipelining in the epilogue)
__device__ __forceinline__ void tmem_ld8_async(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}

// -DTACTOR_PROF: per-warp wait / work cycle counters of CTA 0 (development build only: python -m mop_truss_marl_b200.build
// --prof, scripts/actor_prof.py); the counters land behind the error flag: [warp][8] long long at error_flag + 32 ints
#ifdef TACTOR_PROF
#define PROF_DECL long long prof_c[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const long long prof_start = clock64();
#define PROF_WAIT(slot, expr) do { const long long t0_ = clock64(); expr; prof_c[slot] += clock64() - t0_; } while (0)
#define PROF_ADD(slot, v) prof_c[slot] += (v)
#define PROF_NOW() clock64()
// time line of item 1 of CTA 0 (raw SM clock, 32 bits): words [w][48 visits][4] per generator warp, then the issuer's
// [91 chunks][4] at word 4096 and the epilogue warps' [4][7][2] at word 4608, all behind error_flag + 2048 ints
#define PROF_TRACE(word, value_expr) do { if (blockIdx.x == 0 && lane == 0 && P.error_flag) \
    reinterpret_cast<uint32_t*>(P.error_flag + 2048)[word] = (uint32_t)(value_expr); } while (0)
#define PROF_FLUSH() do { if (blockIdx.x == 0 && lane == 0 && P.error_flag) { prof_c[7] = clock64() - prof_start; \
    long long* dst_ = reinterpret_cast<long long*>(P.error_flag + 32) + warp * 8; for (int i_ = 0; i_ < 8; ++i_) dst_[i_] = prof_c[i_]; } } while (0)
#else
#define PROF_DECL
#define PROF_WAIT(slot, expr) do { expr; } while (0)
#define PROF_ADD(slot, v) do { } while (0)
#define PROF_NOW() 0ll
#define PROF_TRACE(word, value_expr) do { } while (0)
#define PROF_FLUSH() do { } while (0)
#endif

// NREAL: nodes of a real graph when the tensors are padded to NODES rows per environment (12 in 16: the train/code shapes),
// else NODES -- a compile-time constant, so that the production instantiations keep their shifts in the pooled scramble
template <int NODES, int NREAL = NODES>
__global__ void __launch_bounds__(PTHREADS, 1)
actor_pipe_kernel(const __grid_constant__ Params P) {
  constexpr int NGENW = 4 * NPH, W_ISSUER = NGENW + NEPIW, W_PRODUCER = W_ISSUER + 1;
  constexpr int ENVS = TCM / NODES;
  constexpr int KB = NODES / 16;                             // 16-node column blocks of an environment's adjacency matrix
  static_assert(pipe_smem_bytes<NODES>() <= 232448, "shared memory budget");
  static_assert(NODES == 16 || NODES == 32, "a generator warp's 32 rows are two 16-node environments or one of 32");
  static_assert(KCH == 16 && NCH * KCH >= KH + 1, "16-wide chunks; the tail chunk holds the bias column");
  extern __shared__ __align__(128) unsigned char smem[];
  float* H = reinterpret_cast<float*>(smem + WST * STAGE_BYTES);             // [128][LDH]
  uint32_t* W1f = reinterpret_cast<uint32_t*>(H + TCM * LDH);                // layer-1 A fragments, resident
  float* Pl2 = reinterpret_cast<float*>(W1f + W1F_WORDS);                    // [2][ENVS][208] pooled Pareto embedding of the item / the next item
  float* Xr2 = Pl2 + 2 * ENVS * 208;                                         // [2][128][13] raw x_n rows of the item / the next item
  float* AnT = Xr2 + 2 * TCM * 13;                                           // [N(j)][N(n)] shared A_n, transposed (heads)
  uint32_t* AnF = reinterpret_cast<uint32_t*>(AnT + NODES * NODES);         // [KB * KB blocks][hi | lo][32 lanes][4] mma A fragments of the shared A_n
  float* Wh = AnT + 2 * NODES * NODES;                                           // [2][201][4] head kernels, row 200 = bias
  float* Us = Wh + 2 * 201 * 4;                                              // [2 heads][128][4] head pre-activations
  uint64_t* bars = reinterpret_cast<uint64_t*>(Us + 2 * TCM * 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * MAXST + 8);
  // h_prog[row group]: 32 * item + 8-column blocks of GEMM 4 (the last term of the five-way sum H) the group's epilogue
  // warp has stored; the generators of layer 3 start on a column chunk as soon as their rows of it are there
  volatile int* h_prog = reinterpret_cast<volatile int*>(tmem_slot + 2);
  constexpr int NCB = KH / 8;                                // 25 blocks of 8 accumulator columns

  // the shuffle tells the compiler that `warp` is warp-uniform: role branches become uniform branches
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  // CTAs below split_from own a full 128-row tile.  The tiles of the last, partial wave are cut into split_f pieces of
  // 128 / split_f rows, one CTA each, so that the SMs a partial wave would leave idle share its work: a CTA with fewer
  // live rows runs the same barrier protocol, but the warps of its dead 32-row groups skip their work.
  //
  // PERSISTENT: the grid is one CTA per SM and a CTA walks the work items blockIdx.x, blockIdx.x + gridDim.x, ...; TMEM,
  // barriers and the tile-independent constants are set up once, every barrier parity is derived from chunk / GEMM
  // counters that keep running across items, and the generators start on the next item while the issuer and the
  // epilogue still finish the current one.
  auto item_rows = [&](int item, int& row0, int& rows_here) {
    row0 = item * TCM; rows_here = TCM;
    if (item >= P.split_from) {
      const int j = item - P.split_from;
      rows_here = TCM / P.split_f;
      row0 = (P.split_from + j / P.split_f) * TCM + (j % P.split_f) * rows_here;
    }
  };
  const int M = P.M;
  // W ring (s < WST):  w_full  W chunk landed (TMA tx)    w_empty stage consumed (tcgen05.commit)
  // A ring (s < PAST): a_full  A stage written (one arrive per generator warp of the chunk, 4)
  //                    a_empty stage consumed (commit)
  // acc_full[b] accumulator b complete (commit)   acc_empty[b] drained by the epilogue warps
  static_assert(WST <= MAXST && PAST <= MAXST, "barrier slots");
  const uint32_t w_full = smem_u32(&bars[0]), w_empty = smem_u32(&bars[MAXST]);
  const uint32_t a_full = smem_u32(&bars[2 * MAXST]), a_empty = smem_u32(&bars[3 * MAXST]);
  const uint32_t acc_full = smem_u32(&bars[4 * MAXST]), acc_empty = smem_u32(&bars[4 * MAXST + 2]);
  const uint32_t x_full = smem_u32(&bars[4 * MAXST + 6]);      // [2] the item's x_n / pooled rows have landed (cp.async arrivals of all generator threads)

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 32) {
    for (int s = 0; s < WST; ++s) {
      mbar_init(w_full + 8 * s, 1);
      mbar_init(w_empty + 8 * s, 1);
    }
    for (int s = 0; s < PAST; ++s) {
      mbar_init(a_full + 8 * s, 4);                         // the four row-group warps of the chunk's phase
      mbar_init(a_empty + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(acc_full + 8 * b, 1);
      mbar_init(acc_empty + 8 * b, NEPIW);
    }
    mbar_init(x_full, NGENW * 32);
    mbar_init(x_full + 8, NGENW * 32);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // item-independent constants: A_n (both orientations), the head kernels and the layer-1 fragment image; the
  // generators stage the per-item data
  if (tid < 4) h_prog[tid] = 0;
  for (int idx = tid; idx < NODES * NODES; idx += PTHREADS) AnT[(idx % NODES) * NODES + idx / NODES] = P.A_n[idx];
  for (int idx = tid; idx < KB * KB * 32; idx += PTHREADS) {
    // fp16 hi/lo A fragments of the 16 x 16 blocks of A_n (block (mt, kb): rows 16 mt.., columns 16 kb..), computed once
    const int blk = idx >> 5, ln = idx & 31, fg = ln >> 2, ft = ln & 3;
    const float* p0 = P.A_n + (16 * (blk / KB) + fg) * NODES + 16 * (blk % KB) + 2 * ft;
    const float2 v[4] = {*reinterpret_cast<const float2*>(p0), *reinterpret_cast<const float2*>(p0 + 8 * NODES),
                         *reinterpret_cast<const float2*>(p0 + 8), *reinterpret_cast<const float2*>(p0 + 8 * NODES + 8)};
    bool badn = false;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t hi, lo;
      split2(v[i].x, v[i].y, hi, lo);
      AnF[((blk * 2 + 0) * 32 + ln) * 4 + i] = hi;
      AnF[((blk * 2 + 1) * 32 + ln) * 4 + i] = lo;
      badn = badn || !(fabsf(v[i].x) <= F16_MAX) || !(fabsf(v[i].y) <= F16_MAX);
    }
    if (badn && P.error_flag) atomicOr(P.error_flag, 2);
  }
  for (int idx = tid; idx < 2 * 201; idx += PTHREADS) {
    const int hd = idx / 201, k = idx % 201;
    reinterpret_cast<float4*>(Wh)[idx] = (k < KH) ? __ldg(reinterpret_cast<const float4*>(P.w_head[hd] + (size_t)k * 208))
                                                  : __ldg(reinterpret_cast<const float4*>(P.b_head[hd]));
  }
  for (int idx = tid; idx < W1F_WORDS / 4; idx += PTHREADS)
    reinterpret_cast<uint4*>(W1f)[idx] = __ldg(reinterpret_cast<const uint4*>(P.w1frag) + idx);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  bool ok = true;
  PROF_DECL
  // programmatic dependent launch: the env-step kernel that follows in the stream may be scheduled as soon as SMs free up
  // (it waits in griddepcontrol.wait for this grid to finish before it reads the actions)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < NGENW) {
    // =================================================== generators ===========================================
    const int q = warp & 3, ph = warp >> 2;
    const int g8 = lane >> 2, t4 = lane & 3;                 // mma fragment coordinates
    bool bad = false;                                        // an input / adjacency entry / Z outside the fp16 range, or NaN (the ReLU
                                                             // behind Z would hide it; everything downstream shows up as a
                                                             // non-finite accumulator entry, which the epilogue checks)
    // asynchronous copy of one item's x_n rows and pooled rows into buffer `buf` (all generator threads take part)
    auto stage_item = [&](int item_s, int buf) {
      int row0s, rows_s;
      item_rows(item_s, row0s, rows_s);
      const long long xbytes = (long long)M * 13 * 4;        // bytes of x_n that exist
      for (int idx = tid; idx < TCM * 13 / 4; idx += NGENW * 32) {
        const long long off = (long long)row0s * 13 * 4 + (long long)idx * 16;
        const long long left = xbytes - off;
        const int nbytes = left >= 16 ? 16 : (left > 0 ? (int)left : 0);
        const uint32_t dst = smem_u32(Xr2 + buf * TCM * 13 + idx * 4);
        const char* src = reinterpret_cast<const char*>(P.x_n) + (nbytes > 0 ? off : 0);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
      }
      const int env0s = row0s / NODES;
      for (int idx = tid; idx < ENVS * 52; idx += NGENW * 32) {
        const int env = env0s + idx / 52;
        const int nbytes = (env * NODES < M) ? 16 : 0;
        const uint32_t dst = smem_u32(Pl2 + buf * ENVS * 208 + idx * 4);
        const char* src = reinterpret_cast<const char*>(P.pooled) + (nbytes ? ((size_t)env * 208 * 4 + (size_t)(idx % 52) * 16) : 0);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
      }
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(x_full + 8 * buf) : "memory");
      // the three per-environment adjacency tensors of that item are read straight from global memory: pull their
      // lines into L2 now
      if (row0s + TCM <= M) {
        constexpr int LINES = ENVS * NODES * NODES * 4 / 128;
        for (int idx = tid; idx < 3 * LINES; idx += NGENW * 32) {
          const int arr = idx / LINES, line = idx % LINES;
          const float* base = (arr == 0 ? P.A_s : arr == 1 ? P.A_ts : P.A_cs) + (size_t)env0s * NODES * NODES;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(base) + 128 * line));
        }
      }
    };
    const float w1si0 = __ldg(P.wscale_inv + NGEMM), w1si1 = __ldg(P.wscale_inv + NGEMM + 1), w1si2 = __ldg(P.wscale_inv + NGEMM + 2);
    for (int item = blockIdx.x, it = 0; item < P.n_items; item += gridDim.x, ++it) {
      int row0, rows_here;
      item_rows(item, row0, rows_here);
      const int env0 = row0 / NODES;
      const uint32_t ubase = (uint32_t)it * (uint32_t)(NGEMM * NCH);
      // per-item data (x_n rows, pooled rows): double-buffered; the copies of THIS item were issued one item ago
      // (cp.async, 16 bytes each, zero-filled past the batch), so the item starts without global latency.
      // No rendezvous of the generator warps: the buffer's mbarrier completes when the copies of all generator threads
      // have landed, and the buffer being refilled (item it-1's) is free because no warp can be more than PAST chunks behind.
      if (it == 0) {
        asm volatile("griddepcontrol.wait;" ::: "memory");      // the Pareto-branch kernel (pooled) and everything before it are done
        stage_item(item, 0);
      }
      if (item + (int)gridDim.x < P.n_items) stage_item(item + (int)gridDim.x, (it + 1) & 1);
      PROF_WAIT(0, ok = mbar_wait(x_full + 8 * (it & 1), (uint32_t)((it >> 1) & 1)) && ok);
      const float* Xraw = Xr2 + (it & 1) * TCM * 13;
      const float* Pl = Pl2 + (it & 1) * ENVS * 208;
      // HALF-LIVE piece (16-node graphs, a tile of the last wave cut in two): its four environments sit one per 32-row
      // group (tile rows 32 e .. 32 e + 15 = environment e), so that every generator warp carries 16 rows -- half of a full
      // tile's tensor-core and conversion work per chunk -- instead of two warps carrying 32 and two idling: the piece's
      // chunks are then paced by the tcgen05 MMAs rather than by the generators
      const bool hl = (NODES == 16) && P.split_f == 2 && item >= P.split_from;
      if (!hl && 32 * q >= rows_here) {
        // dead row group of a split tile: keep the barrier protocol going, produce nothing (the tensor core reads
        // whatever these TMEM lanes hold; rows are independent and the epilogue never looks at them)
        for (int uu = 0; uu < NGEMM * NCH; ++uu) {
          const uint32_t u = ubase + (uint32_t)uu, sa = u % PAST;
          if ((int)(u % NPH) != ph) continue;
          if (u >= PAST) PROF_WAIT(3, ok = mbar_wait(a_empty + 8 * sa, ((u / PAST) - 1) & 1) && ok);
          __syncwarp();
          if (lane == 0) mbar_arrive(a_full + 8 * sa);
        }
        continue;
      }
      // The warp's 32 rows are two 16-row blocks mt = 0, 1.  NODES = 16: block mt is environment 2q + mt and mixes with
      // itself only (KB = 1); NODES = 32: both blocks belong to environment q and every (mt, kb) pair of 16 x 16 sub-blocks of
      // the adjacency matrix takes part.  kr(mt, kb) = the 16-row block of the warp that holds the k rows of the pair.
      // HL (half-live piece, see above): block 0 only, environment q.
      auto item_body = [&](auto hl_tag) {
      constexpr bool HL = decltype(hl_tag)::value;
      constexpr int MT = HL ? 1 : 2;                           // live 16-row blocks of the warp
      auto kr_of = [](int mt, int kb) { return NODES == 16 ? mt : kb; };
      // the 16 x 16 block (rows nb.., columns 16 kb..) of a row-major [N][N] matrix in global memory, as the four float2 of this
      // lane's A fragment
      auto adj_load = [&](const float* base, int mt, int kb, float2* v) {
        const int nb = (16 * mt) % NODES;
        const float* p0 = base + (nb + g8) * NODES + 16 * kb + 2 * t4;
        v[0] = __ldg(reinterpret_cast<const float2*>(p0)); v[1] = __ldg(reinterpret_cast<const float2*>(p0 + 8 * NODES));
        v[2] = __ldg(reinterpret_cast<const float2*>(p0 + 8)); v[3] = __ldg(reinterpret_cast<const float2*>(p0 + 8 * NODES + 8));
      };
      // ... split into fp16 hi/lo fragments (range / NaN check: the sum of the eight entries is finite iff every entry is)
      auto adj_split = [&](const float2* v, uint32_t* hi, uint32_t* lo) {
        const float m = fmaxf(fmaxf(fmaxf(fabsf(v[0].x), fabsf(v[0].y)), fmaxf(fabsf(v[1].x), fabsf(v[1].y))),
                              fmaxf(fmaxf(fabsf(v[2].x), fabsf(v[2].y)), fmaxf(fabsf(v[3].x), fabsf(v[3].y))));
        const float sum = ((v[0].x + v[0].y) + (v[1].x + v[1].y)) + ((v[2].x + v[2].y) + (v[3].x + v[3].y));
        bad = bad || !(m <= F16_MAX) || (sum != sum);
        split2(v[0].x, v[0].y, hi[0], lo[0]); split2(v[1].x, v[1].y, hi[1], lo[1]);
        split2(v[2].x, v[2].y, hi[2], lo[2]); split2(v[3].x, v[3].y, hi[3], lo[3]);
      };
      // fragments of the shared A_n: precomputed image (hi | lo) in shared memory
      auto an_frag = [&](int mt, int kb, uint32_t* hi, uint32_t* lo) {
        const int blk = (NODES == 16) ? 0 : 2 * mt + kb;
        const uint4 h = *reinterpret_cast<const uint4*>(AnF + ((blk * 2 + 0) * 32 + lane) * 4);
        const uint4 l = *reinterpret_cast<const uint4*>(AnF + ((blk * 2 + 1) * 32 + lane) * 4);
        hi[0] = h.x; hi[1] = h.y; hi[2] = h.z; hi[3] = h.w;
        lo[0] = l.x; lo[1] = l.y; lo[2] = l.z; lo[3] = l.w;
      };
      // per-environment adjacency tensor of GEMM g (nullptr: the shared A_n); its raw entries are fetched one such GEMM ahead
      // (GEMM 1's at the start of the item), so that no global latency sits between two GEMMs
      auto adj_tensor = [&](int g) -> const float* { return (g == 1) ? P.A_ts : (g == 2) ? P.A_cs : (g == 3 || g == 6) ? P.A_s : nullptr; };
      float2 araw[2][KB][4];
      auto fetch_adj = [&](int g) {
        const float* t = adj_tensor(g);
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          int env = env0 + (HL ? q : (32 * q + 16 * mt) / NODES);   // clamped into the batch (rows past the batch are never written)
          env = env * NODES < M ? env : (M / NODES - 1);
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) adj_load(t + (size_t)env * NODES * NODES, mt, kb, araw[mt][kb]);
        }
      };
      fetch_adj(1);
      // ---- Z = A_n . x_n (gcn_l1_1..3 share input and adjacency), kept as the B fragments of [Z, 1]^T:
      //      zfr[8-row block of the warp][hi | lo][c 0..7 | c 8..15 (c = 13: the constant 1 that multiplies the bias row)] ----
      uint32_t zfr[4][2][2];
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        float z[2][4];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) z[nt][0] = z[nt][1] = z[nt][2] = z[nt][3] = 0.f;
#pragma unroll
        for (int kb = 0; kb < KB; ++kb) {
          uint32_t ahi[4], alo[4];
          an_frag(mt, kb, ahi, alo);
          const float* xr = Xraw + ((HL ? 16 : 32) * q + 16 * kr_of(mt, kb) + 2 * t4) * 13;   // rows of the staged block (contiguous from row0)
#pragma unroll
          for (int nt = 0; nt < 2; ++nt) {
            const int c = 8 * nt + g8;
            float x00 = 0.f, x01 = 0.f, x10 = 0.f, x11 = 0.f;
            if (c < 13) { x00 = xr[c]; x01 = xr[13 + c]; x10 = xr[8 * 13 + c]; x11 = xr[9 * 13 + c]; }
            bad = bad || !(fabsf(x00) <= F16_MAX) || !(fabsf(x01) <= F16_MAX) || !(fabsf(x10) <= F16_MAX) || !(fabsf(x11) <= F16_MAX);
            uint32_t bhi[2], blo[2];
            split2(x00, x01, bhi[0], blo[0]);
            split2(x10, x11, bhi[1], blo[1]);
            hmma_split(z[nt], ahi, alo, bhi, blo);
          }
        }
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int i = 0; i < 4; ++i) bad = bad || !(fabsf(z[nt][i]) <= F16_MAX);
        if (t4 == 2) { z[1][1] = 1.f; z[1][3] = 1.f; }       // column c = 13
        split2(z[0][0], z[0][1], zfr[2 * mt][0][0], zfr[2 * mt][1][0]);
        split2(z[1][0], z[1][1], zfr[2 * mt][0][1], zfr[2 * mt][1][1]);
        split2(z[0][2], z[0][3], zfr[2 * mt + 1][0][0], zfr[2 * mt + 1][1][0]);
        split2(z[1][2], z[1][3], zfr[2 * mt + 1][0][1], zfr[2 * mt + 1][1][1]);
      }
      // Hand-off of an A stage, decoupled from the chunk that filled it: the stage is acquired (a_empty) only right before
      // its tcgen05.st, and published (wait::st, fence, arrive on a_full) in the middle of the NEXT chunk's arithmetic, so
      // neither the barrier round trip nor the tensor-memory store latency sits on the warp's dependent chain.
      int pending = -1;                                        // stage written but not yet published
      auto hand_off = [&]() {
        if (pending < 0) return;                               // warp-uniform
        PROF_WAIT(4, asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"));
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full + 8 * pending);
        pending = -1;
      };
      uint32_t afr[2][KB][2][4];                               // [mt][kb][hi | lo][a0..a3] of the GEMM's adjacency matrix
      for (int g = 0; g < NGEMM; ++g) {
        // ---- per-GEMM setup: adjacency fragments; pull the next GEMM's rows towards the SM ----
        if (g == 1 || g == 2 || g == 3 || g == 6) {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) adj_split(araw[mt][kb], afr[mt][kb][0], afr[mt][kb][1]);
          if (g < 6) fetch_adj(g < 3 ? g + 1 : 6);
        } else {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) an_frag(mt, kb, afr[mt][kb][0], afr[mt][kb][1]);
        }
        const float w1si = (g == 0) ? w1si0 : (g <= 2 ? w1si1 : w1si2);
        const uint32_t* w1f = W1f + ((g == 0) ? 0 : (g <= 2 ? 1 : 2)) * (NCH * 2 * 32 * 4);   // gcn_l1_1 | gcn_l1_2 (g = 1, 2) | gcn_l1_3
        // ---- this warp's chunks of the GEMM ----
        for (int c = 0; c < NCH; ++c) {
          const uint32_t u = ubase + (uint32_t)(g * NCH + c), sa = u % PAST;
          if ((int)(u % NPH) != ph) continue;                  // another phase's warps own this chunk
          const int k0 = c * KCH;
          const long long prof_t1 = PROF_NOW();
          const int prof_v = (g * NCH + c) / NPH;
          if (it == 1) PROF_TRACE((warp * 48 + prof_v) * 4 + 0, prof_t1);
          // the five-way sum H is handed over row group by row group, 16 columns at a time: the epilogue warp of this
          // warp's rows publishes how many of its 8-column blocks of GEMM 4 are stored (h_prog), so layer 3 starts on
          // column chunk c as soon as blocks 2c, 2c + 1 are there instead of after the whole drain
          if (g == 5) {
            const int want = it * 32 + min(2 * c + 2, NCB);
            const long long t0_ = PROF_NOW();
            uint32_t spin = 0;
            while (h_prog[q] < want && ++spin < SPIN_LIMIT) { }
            ok = ok && spin < SPIN_LIMIT;
            __threadfence_block();
            PROF_ADD(1, PROF_NOW() - t0_);
          }
          // X fragments of the chunk: xb[16-row block][8-feature half][hi | lo][rows 2t.. | rows 8 + 2t..]
          uint32_t xb[2][2][2][2];
          if (g <= 3) {
            // layer 1 on the tensor core: X^T [16 features x 8 rows] = relu([W1k ; b1k]^T . [Z, 1]^T) XPRE / S for the four
            // 8-row blocks; accumulator element (feature g8 (+8), rows 2t, 2t+1) is exactly what the mix needs as B fragment
            const uint4 wh = *reinterpret_cast<const uint4*>(w1f + ((c * 2 + 0) * 32 + lane) * 4);
            const uint4 wl = *reinterpret_cast<const uint4*>(w1f + ((c * 2 + 1) * 32 + lane) * 4);
            const uint32_t whi[4] = {wh.x, wh.y, wh.z, wh.w}, wlo[4] = {wl.x, wl.y, wl.z, wl.w};
#pragma unroll
            for (int ntr = 0; ntr < 2 * MT; ++ntr) {
              float xt[4] = {0.f, 0.f, 0.f, 0.f};
              hmma_split(xt, whi, wlo, zfr[ntr][0], zfr[ntr][1]);
#pragma unroll
              for (int i = 0; i < 4; ++i) xt[i] = fmaxf(xt[i] * w1si, 0.f);
              split2(xt[0], xt[1], xb[ntr >> 1][0][0][ntr & 1], xb[ntr >> 1][0][1][ntr & 1]);
              split2(xt[2], xt[3], xb[ntr >> 1][1][0][ntr & 1], xb[ntr >> 1][1][1][ntr & 1]);
            }
          } else {
#pragma unroll
            for (int kr = 0; kr < MT; ++kr)
#pragma unroll
              for (int nt = 0; nt < 2; ++nt) {
                const int feat = k0 + 8 * nt + g8;
                float v[2][2] = {{0.f, 0.f}, {0.f, 0.f}};        // [rows 2t.. | 8 + 2t..][row, row + 1]
                if (feat < KH) {
#pragma unroll
                  for (int b = 0; b < 2; ++b)
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                      const int r = 32 * q + 16 * kr + 8 * b + 2 * t4 + i;
                      if (g == 4) {
                        // the reference's stack-and-reshape scramble: x14b[b,n,h] = pooled[b,(n*200+h)/N] (truss2D_RL.py:89-95)
                        v[b][i] = (NREAL == NODES || (r % NODES) < NREAL) ? Pl[(HL ? q : r / NODES) * 208 + ((r % NODES) * KH + feat) / NREAL] : 0.f;   // (padding rows of a 12-in-16 graph: 0)
                      } else {
                        v[b][i] = H[r * LDH + feat];             // layer 3: rows of the five-way sum
                      }
                    }
                }
                split2(v[0][0], v[0][1], xb[kr][nt][0][0], xb[kr][nt][1][0]);
                split2(v[1][0], v[1][1], xb[kr][nt][0][1], xb[kr][nt][1][1]);
              }
          }
          PROF_ADD(5, PROF_NOW() - prof_t1);
          if (it == 1) PROF_TRACE((warp * 48 + prof_v) * 4 + 1, PROF_NOW());
          hand_off();                                          // publish the previous chunk's stage
          const long long prof_t2 = PROF_NOW();
          // ---- Y = A_g . X on the tensor core, split, store from the accumulator layout ----
          uint32_t oh[2][4], ol[2][4];
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
              float y[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
              for (int kb = 0; kb < KB; ++kb) {
                const int kr = kr_of(mt, kb);
                hmma_split(y, afr[mt][kb][0], afr[mt][kb][1], xb[kr][nt][0], xb[kr][nt][1]);
              }
              // column 200 of A is the constant that multiplies the bias row of the W image: the factor every entry of
              // Y carries, XPRE in layer 2, HPRE in layer 3 (columns 201..207 are zero because X is)
              if (k0 + 8 * nt == KH && t4 == 0) { y[0] = (g <= 4) ? XPRE : HPRE; y[2] = y[0]; }
              split2(y[0], y[1], oh[mt][2 * nt], ol[mt][2 * nt]);              // lane g8,     column 4 nt + t4
              split2(y[2], y[3], oh[mt][2 * nt + 1], ol[mt][2 * nt + 1]);      // lane g8 + 8, column 4 nt + t4
            }
          PROF_ADD(6, PROF_NOW() - prof_t2);
          if (it == 1) PROF_TRACE((warp * 48 + prof_v) * 4 + 2, PROF_NOW());
          if (u >= PAST) PROF_WAIT(2, ok = mbar_wait(a_empty + 8 * sa, ((u / PAST) - 1) & 1) && ok);        // chunk u-PAST consumed
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            const uint32_t lane_sel = (uint32_t)(32 * q + 16 * mt) << 16;
            tmem_st_16x128b_x2(tmem_base + lane_sel + (uint32_t)(TM_AHI + ACOLS * sa), oh[mt]);
            tmem_st_16x128b_x2(tmem_base + lane_sel + (uint32_t)(TM_ALO + ACOLS * sa), ol[mt]);
          }
          pending = (int)sa;
          if (it == 1) PROF_TRACE((warp * 48 + prof_v) * 4 + 3, PROF_NOW());
          // the tensor core runs dry at the head of every GEMM (the generators paid the GEMM's set-up, and layer 3 waited for
          // the five-way sum): publish its first chunks at once instead of in the middle of the warp's next chunk
          if (c < NPH) hand_off();
        }
        hand_off();                                            // the accumulator of this GEMM must not wait for the next one
      }
      };  // item_body
      if constexpr (NODES == 16) {
        if (hl) item_body(std::true_type{});
        else item_body(std::false_type{});
      } else {
        item_body(std::false_type{});
      }
    }  // items
    if (bad && P.error_flag) atomicOr(P.error_flag, 2);        // an input left the fp16 range (or NaN)
  } else if (warp < NGENW + NEPIW) {
    // =================================================== epilogue =============================================
    const int q = warp & 3;                                    // row group
    const int r = 32 * q + lane;
    const int n = r % NODES;
    const int lane_env0 = lane & ~(NODES - 1);
    float nonfinite = 0.f;                                     // stays 0 while every accumulator entry is finite (x * 0 is NaN otherwise)
    for (int item = blockIdx.x, it = 0; item < P.n_items; item += gridDim.x, ++it) {
      int row0, rows_here;
      item_rows(item, row0, rows_here);
      const bool hl = (NODES == 16) && P.split_f == 2 && item >= P.split_from;   // half-live piece: lanes 0..15 of every row group
      const bool live = hl || 32 * q < rows_here;              // dead row group of a split tile: barriers only
      const float nonfinite_in = nonfinite;
      for (int g = 0; g < NGEMM; ++g) {
        const int G = it * NGEMM + g, b = G & 1;               // GEMM counter across items: accumulator and parity
        PROF_WAIT(0, ok = mbar_wait(acc_full + 8 * b, (uint32_t)((G >> 1) & 1)) && ok);
        if (!live) {
          __syncwarp();
          if (lane == 0) mbar_arrive(acc_empty + 8 * b);
          continue;
        }
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const long long prof_t1 = PROF_NOW();
        if (it == 1) PROF_TRACE(4608 + (q * 7 + g) * 2, prof_t1);
        const uint32_t tacc = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(b ? TM_ACC1 : 0);
        const float wsi = __ldg(P.wscale_inv + g);             // undoes the power-of-two scale folded into W and the operand factors (exact)
        float* hrow = H + r * LDH;
        const float* wh = Wh + (g >= 5 ? g - 5 : 0) * 201 * 4; // only used for g >= 5
        float u0 = 0.f, u1 = 0.f, u2 = 0.f;
        uint32_t vr[2][8];
        tmem_ld8_async(tacc, vr[0]);
#pragma unroll 2
        for (int i = 0; i < NCB; ++i) {
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          float v[8];
#pragma unroll
          for (int t = 0; t < 8; ++t) v[t] = __uint_as_float(vr[i & 1][t]);
          if (i + 1 < NCB) tmem_ld8_async(tacc + (uint32_t)(8 * (i + 1)), vr[(i + 1) & 1]);   // in flight while block i is processed
          // an operand that left the fp16 range (|A.X| > 65504 became inf in the split) or a NaN shows up as a non-finite
          // accumulator entry here, before the ReLU can hide it: one FFMA per entry instead of range tracking in the generators
#pragma unroll
          for (int t = 0; t < 8; ++t) nonfinite = fmaf(v[t], 0.f, nonfinite);
          // relu(D / S) with the bias riding along as row 200 of the W image; 1/S is a power of two, so relu(D) (1/S) + H in one
          // FFMA gives the bits of relu(D / S) + H
          if (g <= 4) {
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = fmaxf(v[t], 0.f);
            float4* dst = reinterpret_cast<float4*>(hrow + 8 * i);
            float4 o0 = make_float4(0.f, 0.f, 0.f, 0.f), o1 = o0;
            if (g > 0) { o0 = dst[0]; o1 = dst[1]; }
            dst[0] = make_float4(fmaf(v[0], wsi, o0.x), fmaf(v[1], wsi, o0.y), fmaf(v[2], wsi, o0.z), fmaf(v[3], wsi, o0.w));
            dst[1] = make_float4(fmaf(v[4], wsi, o1.x), fmaf(v[5], wsi, o1.y), fmaf(v[6], wsi, o1.z), fmaf(v[7], wsi, o1.w));
            if (g == 4) {                                      // H is complete in these 8 columns of this warp's rows
              __threadfence_block();
              __syncwarp();
              if (lane == 0) h_prog[q] = it * 32 + i + 1;
            }
          } else {
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = fmaxf(v[t] * wsi, 0.f);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              const float4 w = *reinterpret_cast<const float4*>(wh + (8 * i + t) * 4);
              u0 = fmaf(v[t], w.x, u0); u1 = fmaf(v[t], w.y, u1); u2 = fmaf(v[t], w.z, u2);
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        PROF_ADD(1, PROF_NOW() - prof_t1);
        if (it == 1) PROF_TRACE(4608 + (q * 7 + g) * 2 + 1, PROF_NOW());
        if (lane == 0) mbar_arrive(acc_empty + 8 * b);
        if (g >= 5) {
          // output heads (truss2D_RL.py:121-125): sigmoid(A_n (x3 W4) + b4); the 16/32 rows of an environment are
          // lanes of this warp, whose x3 W4 rows meet in shared memory
          const int hd = g - 5, nout = 2 + hd;
          float* us = Us + hd * TCM * 4;                       // [128][4]
          *reinterpret_cast<float4*>(us + r * 4) = make_float4(u0, u1, u2, 0.f);
          __syncwarp();
          float o[3] = {wh[KH * 4 + 0], wh[KH * 4 + 1], wh[KH * 4 + 2]};
          for (int j = 0; j < NODES; ++j) {
            const float a = AnT[j * NODES + n];
            const float4 uj = *reinterpret_cast<const float4*>(us + (32 * q + lane_env0 + j) * 4);
            o[0] = fmaf(a, uj.x, o[0]); o[1] = fmaf(a, uj.y, o[1]); o[2] = fmaf(a, uj.z, o[2]);
          }
          __syncwarp();
          const int row = row0 + (hl ? 16 * q + lane : r);
          if (row < M && (!hl || lane < 16) && (NREAL == NODES || n < NREAL)) {      // padding rows of a 12-in-16 graph are not outputs
            const size_t orow = (NREAL == NODES) ? (size_t)row : (size_t)(row / NODES) * NREAL + n;
            float* dst = (hd == 0 ? P.geo : P.topo) + orow * nout;
            uint64_t seed = P.seed, call = P.call;
            if (P.noise && P.seed_call) { seed = P.seed_call[0]; call += P.seed_call[1]; }
            for (int t = 0; t < nout; ++t) {
              float v = 1.f / (1.f + expf(-o[t]));
              if (P.noise) v = ou_step(v, P.mu, P.theta, P.sigma, seed, call, (uint64_t)(hd + 1), (uint64_t)orow * nout + t);
              dst[t] = v;
            }
          }
        }
      }
      if (hl && lane >= 16) nonfinite = nonfinite_in;          // the dead lanes of a half-live piece multiply whatever their TMEM rows hold
    }  // items
    if (!(nonfinite == 0.f) && P.error_flag) atomicOr(P.error_flag, 2);   // an activation left the fp16 range (or NaN)
  } else if (warp == W_ISSUER) {
    // =================================================== MMA issuer ===========================================
    // The whole warp walks the chunk sequence converged (all lanes poll the barriers); ONE elected lane issues the three
    // MMAs and the commits of a chunk.  Stage indices and barrier parities are running counters (no division), and the
    // shared-memory descriptor of a W stage is the stage-0 descriptor plus a constant (its address field counts 16-byte
    // units), so a chunk costs the issuer a few dozen instructions: it is the one serial thread every chunk passes through
    // (the first form -- one lane inside `if (lane == 0)`, u % WST / u % PAST, a switch over per-stage descriptors -- made
    // ptxas wrap every tcgen05 instruction in an elect / branch sequence: ~140 instructions and ~760 cycles per chunk).
    const uint64_t d_hi0 = make_desc(smem_u32(smem), B_LBO);
    constexpr uint64_t D_STAGE = (uint64_t)(STAGE_BYTES >> 4), D_LO = (uint64_t)((NKB * B_LBO) >> 4);
    static_assert((WST * STAGE_BYTES >> 4) < 0x4000, "the W ring must stay inside the descriptor's 14-bit address field");
    uint32_t sw = 0, pw = 0, sa = 0, pa = 0, G = 0;
    for (int item = blockIdx.x; item < P.n_items; item += gridDim.x) {
      const bool prof_tr = (G == (uint32_t)NGEMM);            // item 1 of this CTA
      for (int g = 0; g < NGEMM; ++g, ++G) {
        const uint32_t b = G & 1u;
        const uint32_t dacc = tmem_base + (b ? (uint32_t)TM_ACC1 : 0u);
        if (G >= 2) {                                          // the epilogue of GEMM G-2 has drained this accumulator
          PROF_WAIT(2, ok = mbar_wait_cluster(acc_empty + 8 * b, ((G >> 1) - 1u) & 1u) && ok);
        }
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) {
          PROF_WAIT(0, ok = mbar_wait(a_full + 8 * sa, pa) && ok);
          if (prof_tr) PROF_TRACE(4096 + (g * NCH + c) * 4 + 0, PROF_NOW());
          PROF_WAIT(1, ok = mbar_wait(w_full + 8 * sw, pw) && ok);
          if (prof_tr) PROF_TRACE(4096 + (g * NCH + c) * 4 + 1, PROF_NOW());
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          if (elect_one()) {
            const uint32_t a_hi = tmem_base + (uint32_t)TM_AHI + (uint32_t)ACOLS * sa, a_lo = tmem_base + (uint32_t)TM_ALO + (uint32_t)ACOLS * sa;
            const uint64_t d_hi = d_hi0 + D_STAGE * sw, d_lo = d_hi + D_LO;
            mma_split(dacc, a_hi, d_hi, c != 0);               // Yhi.Whi + Yhi.Wlo + Ylo.Whi (the tail chunk is zero-padded)
            mma_split(dacc, a_hi, d_lo, 1);
            mma_split(dacc, a_lo, d_hi, 1);
            mma_commit(w_empty + 8 * sw);
            mma_commit(a_empty + 8 * sa);
            if (c + 1 == NCH) mma_commit(acc_full + 8 * b);
          }
          __syncwarp();
          if (prof_tr) PROF_TRACE(4096 + (g * NCH + c) * 4 + 2, PROF_NOW());
          if (++sw == (uint32_t)WST) { sw = 0; pw ^= 1u; }
          if (++sa == (uint32_t)PAST) { sa = 0; pa ^= 1u; }
        }
      }
    }  // items
    __syncwarp();
  } else {
    // =================================================== W producer ===========================================
    if (lane == 0) {
      for (int item = blockIdx.x, it = 0; item < P.n_items; item += gridDim.x, ++it)
        for (int g = 0; g < NGEMM; ++g)
          for (int c = 0; c < NCH; ++c) {
            const uint32_t u = (uint32_t)it * (uint32_t)(NGEMM * NCH) + (uint32_t)(g * NCH + c), s = u % WST;
            if (u >= WST) PROF_WAIT(0, ok = mbar_wait(w_empty + 8 * s, ((u / WST) - 1) & 1) && ok);       // chunk u-WST consumed
            const uint32_t bytes = (uint32_t)STAGE_BYTES;                                    // hi then lo
            const unsigned char* src = reinterpret_cast<const unsigned char*>(P.wimg[g]) + (size_t)c * bytes;
            mbar_expect_tx(w_full + 8 * s, bytes);
            bulk_g2s(smem_u32(smem + s * STAGE_BYTES), src, bytes, w_full + 8 * s);
          }
    }
    __syncwarp();
  }

  PROF_FLUSH();
  if (!ok && P.error_flag) atomicOr(P.error_flag, 1);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
}

}  // namespace pipe
}  // namespace tc
}  // namespace tactor
